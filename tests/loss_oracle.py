"""
Test helper: CPU restatement of the pairwise-distance branch of BertForDiffusion._get_loss_terms
(/root/reference/foldingdiff/modelling.py:616-677) with nerf.nerf_build_batch (nerf.py:207-292, place_dihedral's torch
branch :145-204) and losses.pairwise_dist_loss (losses.py:66-150), in plain torch at a chosen precision.

The reference itself mixes precisions (float64 coordinates from its numpy start frame, float32 bond terms); here every
step runs in `dtype`, so the fp32 and fp64 versions bracket the arithmetic and their distance measures how much of a
difference on a given input is rounding.  tests/golden/ref_pdist.npz holds the unmodified reference's answers.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from oracle.nerf import CA_C_LENGTH, C_INIT, C_N_LENGTH, CA_INIT, N_CA_LENGTH, N_INIT

PDIST_COLUMNS = ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"]


def place_dihedral(a, b, c, bond_angle, bond_length, torsion):
    """nerf.py:145-204 (use_torch=True) on (B, 3) points and (B, 1) angles."""
    unit = lambda x: x / torch.linalg.norm(x, dim=-1, keepdim=True)
    ab = b - a
    bc = unit(c - b)
    n = unit(torch.linalg.cross(ab, bc, dim=-1))
    nbc = torch.linalg.cross(n, bc, dim=-1)
    m = torch.stack([bc, nbc, n], dim=-1)
    d = torch.stack([-bond_length * torch.cos(bond_angle),
                     bond_length * torch.cos(torsion) * torch.sin(bond_angle),
                     bond_length * torch.sin(torsion) * torch.sin(bond_angle)], dim=a.ndim - 1).type(m.dtype)
    return torch.matmul(m, d).reshape(c.shape) + c


def nerf_build_batch(angles: torch.Tensor, names: Sequence[str], dtype=torch.float64) -> torch.Tensor:
    """nerf.py:207-292: (B, N, F) angles with columns `names` -> (B, 3N, 3) coordinates in `dtype`, uncentred."""
    a = angles.to(dtype)
    col = {k: a[:, :, list(names).index(k)] for k in PDIST_COLUMNS}
    B = a.shape[0]
    coords = torch.from_numpy(np.array([N_INIT, CA_INIT, C_INIT])).to(dtype).repeat(B, 1, 1)
    phi, psi, omega = col["phi"][:, 1:], col["psi"][:, :-1], col["omega"][:, :-1]
    pts = [coords[:, 0], coords[:, 1], coords[:, 2]]
    for i in range(phi.shape[1]):
        n = place_dihedral(pts[-3], pts[-2], pts[-1], col["CA:C:1N"][:, i:i + 1], C_N_LENGTH, psi[:, i:i + 1])
        ca = place_dihedral(pts[-2], pts[-1], n, col["C:1N:1CA"][:, i:i + 1], N_CA_LENGTH, omega[:, i:i + 1])
        c = place_dihedral(pts[-1], n, ca, col["tau"][:, i:i + 1], CA_C_LENGTH, phi[:, i:i + 1])
        pts += [n, ca, c]
    return torch.stack(pts, dim=1)


def pdist_term(corrupted, eps_hat, known_angles, sqrt_abar, sqrt_1m_abar, coef, lengths, names, dtype=torch.float64):
    """modelling.py:616-677: the pairwise CA-distance term, every step in `dtype` (denoising in fp32 as the reference)."""
    B = corrupted.shape[0]
    denoised = corrupted - sqrt_1m_abar.reshape(B, 1, 1) * eps_hat
    denoised /= sqrt_abar.reshape(B, 1, 1)
    # only the first max(lengths) residues can reach a kept pair: build that prefix (NeRF is a forward recurrence)
    L = int(max(int(l) for l in lengths))
    xa = nerf_build_batch(denoised[:, :L], names, dtype)[:, 1::3]
    xb = nerf_build_batch(known_angles[:, :L], names, dtype)[:, 1::3]
    total, count = torch.zeros((), dtype=dtype), 0
    w = coef.reshape(-1).to(dtype)
    for b in range(B):
        l = int(lengths[b])
        da, db = torch.nn.functional.pdist(xa[b, :l]), torch.nn.functional.pdist(xb[b, :l])
        total = total + (w[b] * (da - db) ** 2).sum()
        count += da.numel()
    return total / count, denoised
