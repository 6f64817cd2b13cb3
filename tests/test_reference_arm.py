"""
The reference arm of bench.py (baseline/reference_arm.py): stock reference loop + sub-modules from baseline/_ref.
tests/golden/ref_loop.npz holds what that arm computed on the inputs below (tests/golden/make_golden_reference.py);
the oracle must reproduce it.
"""
import torch

from conftest import load_golden, mini_state_dict
from oracle import forward as ofwd
from oracle import loop as oloop
from oracle import schedules as osched
from oracle.replay import digest

LOOP_T, LOOP_LENGTHS = 5, [24, 17, 24]


def forward_inputs():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(3, 96, 6, generator=g)
    t = torch.tensor([0, 17, 249])
    mask = torch.ones(3, 96); mask[1, 60:] = 0; mask[2, 33:] = 0
    return x, t, mask


def loop_noise():
    g = torch.Generator().manual_seed(11)
    return oloop.wrap(torch.randn(3, 24, 6, generator=g))


def test_assembled_reference_model_matches_oracle_forward():
    sd, cfg, _, _ = mini_state_dict()
    oracle = ofwd.OracleModel(sd, ofwd.OracleConfig(**cfg), [True] * 6).eval()
    x, t, mask = forward_inputs()
    got = torch.from_numpy(load_golden("ref_loop.npz")["arm_forward"])
    with torch.no_grad():
        want = oracle(x, t, attention_mask=mask)
    err = float((got - want)[mask.bool()].abs().max())
    print(f"reference-assembled model vs oracle forward: {err:.3e}")
    assert err < 2e-6


def test_stock_reference_loop_drives_the_assembled_model_like_the_oracle_loop():
    g = load_golden("ref_loop.npz")
    sd, cfg, _, _ = mini_state_dict()
    oracle = ofwd.OracleModel(sd, ofwd.OracleConfig(**cfg), [True] * 6).eval()
    betas = osched.betas_for("linear", LOOP_T)
    assert digest(betas) == str(g["arm_loop_betas"])
    ref_hist = torch.from_numpy(g["arm_loop_hist"])
    torch.manual_seed(5)
    ora_hist = oloop.p_sample_loop(oracle, LOOP_LENGTHS, loop_noise(), LOOP_T, betas, [True] * 6)
    worst = max(float(oloop.circular_abs_diff(ref_hist[:, i, :l], ora_hist[:, i, :l], [True] * 6).max())
                for i, l in enumerate(LOOP_LENGTHS))
    print(f"stock loop + assembled model vs oracle loop + oracle model, {LOOP_T} steps: {worst:.3e}")
    assert worst < 1e-5
