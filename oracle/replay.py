"""
ORACLE (test infrastructure) - stored answers of the reference for exact comparisons, and model-call replay.

`digest` condenses an array to a SHA-256 of its dtype, shape and bytes: a bit-exact comparison needs nothing more, so
tests/golden/make_golden_reference.py stores digests instead of the arrays where a test compares bit for bit.

A loop compared bit for bit against the reference's loop has to see bit-identical predictions, but a CPU forward pass
is only reproducible to the last bits on the same instruction set (GEMM blocking and reduction order follow the vector
width).  So the generator records every (x, t, mask) -> eps call the reference's loop made (`Recorder`), a test replays
the recorded eps to the restated loop, which must ask with bit-identical inputs in the same order (`Replay`), and the
forward itself is compared with the recorded eps separately, with a tolerance.
"""
from __future__ import annotations

import hashlib
from typing import Dict

import numpy as np
import torch


def digest(a) -> str:
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


class Recorder(torch.nn.Module):
    """Wraps a noise predictor and keeps every call.  A module holding the wrapped model's parameters, so the
    reference's loop (which asks `next(model.parameters()).device`) drives it unmodified."""

    def __init__(self, model: torch.nn.Module, n_inputs: int = 6):
        super().__init__()
        self.model = model
        self.n_inputs = n_inputs
        self.calls = []

    def forward(self, x, t, attention_mask):
        eps = self.model(x, t, attention_mask=attention_mask)
        self.calls.append((digest(x), digest(t), digest(attention_mask), eps.detach().clone()))
        return eps

    def arrays(self, prefix: str) -> Dict[str, np.ndarray]:
        """`<prefix>_calls`, and per call k the input digests `<prefix>_{x,t,mask}_<k>` and the output `<prefix>_eps_<k>`."""
        out = {f"{prefix}_calls": np.array(len(self.calls))}
        for k, (x, t, mask, eps) in enumerate(self.calls):
            out.update({f"{prefix}_x_{k}": np.array(x), f"{prefix}_t_{k}": np.array(t), f"{prefix}_mask_{k}": np.array(mask),
                        f"{prefix}_eps_{k}": eps.numpy()})
        return out


class Replay:
    """Answers the k-th call with the k-th recorded eps, after checking the call's inputs are the recorded ones."""

    def __init__(self, golden, prefix: str, n_inputs: int = 6):
        self.g, self.prefix, self.n_inputs = golden, prefix, n_inputs
        self.total = int(golden[f"{prefix}_calls"])
        self.calls = 0

    def __call__(self, x, t, attention_mask):
        k = self.calls
        assert k < self.total, f"more calls than the {self.total} recorded"
        for name, v in (("x", x), ("t", t), ("mask", attention_mask)):
            assert digest(v) == str(self.g[f"{self.prefix}_{name}_{k}"]), f"call {k}: {name} differs from the recording"
        self.calls += 1
        return torch.from_numpy(self.g[f"{self.prefix}_eps_{k}"]).clone()
