"""
The training objective, forward half: loss terms on the device and the validation loss of a dataset.

Device entry points (include/foldingdiff_b200.h; kernels in csrc/loss.cuh), thin wrappers over the C ABI:
  * `q_sample`     forward noising of a batch (reference datasets.py:772-799, :801-886), torch-given or Philox noise
  * `loss_terms`   the per-feature terms of BertForDiffusion._get_loss_terms (modelling.py:571-604) and their
                   per-chain sums
  * `pdist_loss`   its pairwise-distance term (modelling.py:616-677, losses.py:66-150)
and the evaluation loop:
  * `validation_loss(model, noised_dset, ...)`  what the reference's validation epoch reports (validation_step +
                   validation_epoch_end, modelling.py:719-760) over the unshuffled loader order of bin/train.py:384-394,
                   plus, for an `exhaustive_t` dataset, the loss at every timestep.

There is no CPU path: every call needs CUDA tensors and the library.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native

LOSS_KINDS = {"smooth_l1": 0, "l1": 1}
LOSS_AUTOCORRECT = {"radian_l1_smooth": "smooth_l1"}  # reference modelling.py:235-237
PDIST_COLUMNS = ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev_f32(t: torch.Tensor, device) -> torch.Tensor:
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


def _u8(flags: Sequence[bool]):
    return (C.c_uint8 * len(flags))(*[1 if f else 0 for f in flags])


def q_sample(x0: torch.Tensor, sqrt_abar: torch.Tensor, sqrt_1m_abar: torch.Tensor, is_angular: Sequence[bool],
             var_scale: Sequence[float], z: Optional[torch.Tensor] = None, seed: int = 0, offset: int = 0):
    """
    -> (known_noise, corrupted), both (B, N, F) on x0's device.  `z` (B, N, F) are the caller's standard normals (torch's
    draw: bit-identical to NoisedAnglesDataset.__getitem__); None draws element offset + (b N + n) F + f of the
    library's Philox stream `seed` instead.
    """
    assert x0.is_cuda and x0.dim() == 3
    dev = x0.device
    x0 = _dev_f32(x0, dev)
    B, N, F = x0.shape
    sa, s1m = _dev_f32(sqrt_abar.reshape(-1), dev), _dev_f32(sqrt_1m_abar.reshape(-1), dev)
    assert sa.numel() == B and s1m.numel() == B
    zz = None if z is None else _dev_f32(z, dev)
    assert zz is None or zz.shape == x0.shape
    scales = (C.c_float * F)(*[float(s) for s in var_scale])
    known, corrupted = torch.empty_like(x0), torch.empty_like(x0)
    lib = _native.lib()
    with torch.cuda.device(dev):
        _native.check(lib.fd_q_sample(x0.data_ptr(), B, N, F, sa.data_ptr(), s1m.data_ptr(), scales, _u8(is_angular),
                                      None if zz is None else zz.data_ptr(), int(seed), int(offset), known.data_ptr(),
                                      corrupted.data_ptr(), _stream()), "fd_q_sample")
    return known, corrupted


def loss_terms(eps_hat: torch.Tensor, known_noise: torch.Tensor, attn_mask: torch.Tensor, is_angular: Sequence[bool],
               loss: str = "smooth_l1", circle_penalty: float = 0.0):
    """
    -> (terms (F,), chain_sums (B, 2F + 1) float64): terms[f] is the reference's loss of feature f over the tokens with
    attn_mask != 0; chain_sums[b] holds chain b's loss sums, circle sums and valid-token count.
    """
    assert eps_hat.is_cuda and eps_hat.shape == known_noise.shape
    dev = eps_hat.device
    loss = LOSS_AUTOCORRECT.get(loss, loss)
    if loss not in LOSS_KINDS:
        raise ValueError(f"loss={loss!r}: expected one of {sorted(LOSS_KINDS)}")
    B, N, F = eps_hat.shape
    p, k = _dev_f32(eps_hat, dev), _dev_f32(known_noise, dev)
    m = _dev_f32(attn_mask, dev)
    assert m.shape == (B, N)
    chain = torch.empty(B, 2 * F + 1, dtype=torch.float64, device=dev)
    terms = torch.empty(F, dtype=torch.float32, device=dev)
    lib = _native.lib()
    with torch.cuda.device(dev):
        _native.check(lib.fd_loss_terms(p.data_ptr(), k.data_ptr(), m.data_ptr(), B, N, F, _u8(is_angular),
                                        LOSS_KINDS[loss], float(circle_penalty), chain.data_ptr(), terms.data_ptr(),
                                        _stream()), "fd_loss_terms")
    return terms, chain


def pdist_coefficients(use_pairwise_dist_loss, t: torch.Tensor) -> torch.Tensor:
    """coef_b of modelling.py:648-662: the scalar, or min + (max - min) (T - t_b) / T for the [min, max, T] form."""
    if isinstance(use_pairwise_dist_loss, (list, tuple)):
        min_coef, max_coef, max_timesteps = use_pairwise_dist_loss
        assert 0 < min_coef < max_coef
        coef = min_coef + (max_coef - min_coef) * ((max_timesteps - t) / max_timesteps).to(t.device)
        assert torch.all(coef > 0)
        return coef.reshape(-1).to(torch.float32)
    coef = use_pairwise_dist_loss
    assert coef > 0
    return torch.full((t.shape[0],), float(coef), dtype=torch.float32, device=t.device)


def pdist_loss(corrupted: torch.Tensor, eps_hat: torch.Tensor, known_angles: torch.Tensor, sqrt_abar: torch.Tensor,
               sqrt_1m_abar: torch.Tensor, coef: torch.Tensor, lengths: Sequence[int], ft_names: Sequence[str],
               return_denoised: bool = False):
    """
    -> (loss (), chain_sums (B, 2) float64[, denoised (B, N, F)]): the pairwise CA-distance term between the structure
    of the denoised angles and that of `known_angles` (the batch's zero-centred "angles", as the reference uses them).
    """
    assert corrupted.is_cuda
    dev = corrupted.device
    B, N, F = corrupted.shape
    missing = [c for c in PDIST_COLUMNS if c not in ft_names]
    if missing:
        raise ValueError(f"the pairwise-distance loss needs the features {PDIST_COLUMNS}; missing {missing}")
    cols = (C.c_int32 * 6)(*[list(ft_names).index(c) for c in PDIST_COLUMNS])
    lens = np.ascontiguousarray(np.asarray([int(l) for l in lengths], dtype=np.int32))
    assert lens.size == B
    c, e, a = _dev_f32(corrupted, dev), _dev_f32(eps_hat, dev), _dev_f32(known_angles, dev)
    sa, s1m = _dev_f32(sqrt_abar.reshape(-1), dev), _dev_f32(sqrt_1m_abar.reshape(-1), dev)
    w = _dev_f32(coef.reshape(-1), dev)
    denoised = torch.empty_like(c) if return_denoised else None
    chain = torch.empty(B, 2, dtype=torch.float64, device=dev)
    out = torch.empty((), dtype=torch.float32, device=dev)
    lib = _native.lib()
    with torch.cuda.device(dev):
        _native.check(lib.fd_pdist_loss(c.data_ptr(), e.data_ptr(), a.data_ptr(), sa.data_ptr(), s1m.data_ptr(),
                                        w.data_ptr(), B, N, F, lens.ctypes.data, cols,
                                        None if denoised is None else denoised.data_ptr(), chain.data_ptr(),
                                        out.data_ptr(), _stream()), "fd_pdist_loss")
    return (out, chain, denoised) if return_denoised else (out, chain)


# ------------------------------------------------------------------------------------------------------------------
def _collate(items: List[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
    from torch.utils.data import default_collate
    return default_collate(items)


def _philox_batch(noised_dset, indices: Sequence[int], t_all: torch.Tensor, device, seed: int) -> Dict[str, torch.Tensor]:
    """x0 and t read on the host; the noise is drawn and applied on the device (fd_q_sample, Philox stream `seed`)."""
    inner, key = noised_dset.dset, noised_dset.dset_key
    T = noised_dset.timesteps
    items = []
    for i in indices:
        item_index = i // T if noised_dset.exhaustive_timesteps else i
        items.append(inner[item_index])
    batch = _collate(items)
    x0 = batch[key].to(device)
    B, N, F = x0.shape
    t = t_all[list(indices)].reshape(-1, 1)
    sa = noised_dset.alpha_beta_terms["sqrt_alphas_cumprod"][t.reshape(-1)].to(torch.float32)
    s1m = noised_dset.alpha_beta_terms["sqrt_one_minus_alphas_cumprod"][t.reshape(-1)].to(torch.float32)
    angular = noised_dset.feature_is_angular[key]
    scales = [noised_dset.angular_var_scale if a else noised_dset.nonangular_var_scale for a in angular]
    known, corrupted = q_sample(x0, sa.to(device), s1m.to(device), angular, scales, z=None, seed=seed,
                                offset=int(indices[0]) * N * F)
    batch.update({"corrupted": corrupted, "t": t, "known_noise": known, "sqrt_alphas_cumprod_t": sa,
                  "sqrt_one_minus_alphas_cumprod_t": s1m})
    return batch


@torch.no_grad()
def validation_loss(model, noised_dset, batch_size: int = 512, noise: str = "torch", seed: int = 0,
                    t: Optional[int] = None) -> Dict:
    """
    Evaluate `model` (a modelling.BertForDiffusion on CUDA) on `noised_dset` (a datasets.NoisedAnglesDataset) in the
    reference's unshuffled loader order (bin/train.py:384-394).  Returns
      val_loss      mean over batches of the batch's mean term (what validation_epoch_end reports, modelling.py:753-760)
      terms         {name: mean over batches of that term}  (names: model.ft_names [+ "pairwise_dist_loss"])
      n_items, n_batches
      per_t         (exhaustive_t datasets only) {"t": [0..T-1], "names": [...], "loss": (T, F[+1]) table, "tokens": (T,),
                    "pairs": (T,)}: the feature terms token-weighted over every chain noised to t, the pairwise term
                    pair-weighted - built from the per-chain sums, so re-weighting recovers the whole-set token mean
    noise = "torch": items come from noised_dset.__getitem__ (torch's global generator, as in the reference with
    num_workers = 0; seed the generator first for a reproducible run).  noise = "philox": only x0 and t are read on the
    host (t = the exhaustive index, or drawn from a torch.Generator seeded with `seed`); the noise is element
    (item * N * F + ...) of the library's Philox stream `seed`, independent of batch_size.
    `t` (non-exhaustive datasets only) noises every item to that timestep (__getitem__'s use_t_val).
    """
    if noise not in ("torch", "philox"):
        raise ValueError(f"noise={noise!r}: expected 'torch' or 'philox'")
    if batch_size < 1:
        raise ValueError("batch_size must be >= 1")
    device = next(model.parameters()).device
    n = len(noised_dset)
    T = noised_dset.timesteps
    if t is not None and noised_dset.exhaustive_timesteps:
        raise ValueError("a fixed t cannot be combined with an exhaustive_t dataset")
    if noise == "philox":
        if t is not None:
            t_all = torch.full((n,), int(np.clip(t, 0, T - 1)), dtype=torch.long)
        elif noised_dset.exhaustive_timesteps:
            t_all = torch.arange(n, dtype=torch.long) % T
        else:
            t_all = torch.randint(0, T, (n,), generator=torch.Generator().manual_seed(seed), dtype=torch.long)
    names = list(model.ft_names) + (["pairwise_dist_loss"] if model.pdist_enabled else [])
    batch_means, batch_terms = [], []
    if noised_dset.exhaustive_timesteps:
        F = len(model.ft_names)
        loss_sum = torch.zeros(T, F, dtype=torch.float64)
        circ_sum = torch.zeros(T, F, dtype=torch.float64)
        tokens = torch.zeros(T, dtype=torch.float64)
        pd_sum = torch.zeros(T, dtype=torch.float64)
        pairs = torch.zeros(T, dtype=torch.float64)
    for start in range(0, n, batch_size):
        idx = list(range(start, min(n, start + batch_size)))
        if noise == "torch":
            batch = _collate([noised_dset.__getitem__(i, use_t_val=t) for i in idx])
        else:
            batch = _philox_batch(noised_dset, idx, t_all, device, seed)
        terms, detail = model._loss_terms_detail(batch)
        batch_terms.append(terms)
        batch_means.append(torch.mean(terms))
        if noised_dset.exhaustive_timesteps:
            tb = batch["t"].reshape(-1).to("cpu")
            ch = detail["chain_sums"].to("cpu")
            loss_sum.index_add_(0, tb, ch[:, :F])
            circ_sum.index_add_(0, tb, ch[:, F:2 * F])
            tokens.index_add_(0, tb, ch[:, 2 * F])
            if "pdist_chain_sums" in detail:
                pc = detail["pdist_chain_sums"].to("cpu")
                pd_sum.index_add_(0, tb, pc[:, 0])
                pairs.index_add_(0, tb, pc[:, 1])
    stacked = torch.stack(batch_terms).to("cpu")
    out = {"val_loss": float(torch.mean(torch.stack(batch_means)).item()),
           "terms": {k: float(v) for k, v in zip(names, stacked.mean(dim=0).tolist())},
           "n_items": n, "n_batches": len(batch_terms)}
    if noised_dset.exhaustive_timesteps:
        table = loss_sum / tokens[:, None] + model.circle_lambda * circ_sum / tokens[:, None] * model._circle_mask()[None]
        if model.pdist_enabled:
            table = torch.cat([table, (pd_sum / pairs)[:, None]], dim=1)
        out["per_t"] = {"t": list(range(T)), "names": names, "loss": table.tolist(), "tokens": tokens.tolist(),
                        "pairs": pairs.tolist()}
    return out
