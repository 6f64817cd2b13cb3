"""The oracle (CPU restatement) against the golden vectors written by the reference's own code."""
import numpy as np
import torch

from conftest import load_golden
from oracle import forward as ofwd
from oracle import loop as oloop
from oracle import schedules as osched
from oracle.replay import Replay, digest

SEED = 7344


def test_schedules_bit_exact():
    g = load_golden("schedules.npz")
    for kw in ("cosine", "linear", "quadratic"):
        for T in (1000, 250, 100):
            tab = osched.alpha_tables(osched.betas_for(kw, T))
            for k, v in tab.items():
                assert np.array_equal(v.numpy(), g[f"{kw}_{T}_{k}"]), (kw, T, k)


def test_schedule_known_answers():
    # SURVEY.md A.3 (computed by the reference's own code)
    tab = osched.alpha_tables(osched.betas_for("cosine", 1000))
    assert abs(float(tab["betas"][0]) - 9.99999975e-05) < 1e-12
    assert abs(float(tab["betas"][999]) - 0.999899983) < 1e-7
    assert abs(float(1.0 / torch.sqrt(tab["alphas"][999])) - 99.9917068) < 1e-3
    assert float(tab["posterior_variance"][0]) == 0.0
    for kw in ("cosine", "linear", "quadratic"):  # tests/test_variance_schedules.py:12-40
        b = osched.betas_for(kw, 100)
        assert bool((b[1:] >= b[:-1]).all())


def test_wrap_bit_exact_and_known_answers():
    g = load_golden("wrap.npz")
    vals = torch.from_numpy(g["vals"])
    assert np.array_equal(oloop.wrap(vals.clone(), -np.pi, np.pi).numpy(), g["wrapped"])
    assert np.array_equal(oloop.wrap(vals.clone()).numpy(), g["wrapped_default"])
    assert oloop.wrap(3, -2, 2) == -1  # tests/test_utils.py of the reference
    out = oloop.wrap(torch.tensor([3.5, -3.5, np.pi, 7.0, 100.0], dtype=torch.float32))
    expect = torch.tensor([-2.7831852, 2.7831852, -3.1415927, 0.7168148, -0.5309665])
    assert torch.allclose(out, expect, atol=1e-6)
    w = g["wrapped"]
    assert w.min() >= -np.float32(np.pi) and w.max() < np.pi


def test_sample_noise_bit_exact():
    g = load_golden("noise.npz")
    torch.manual_seed(SEED)
    n1 = oloop.sample_noise(torch.zeros(4, 128, 6), [True] * 6)
    assert np.array_equal(n1.numpy(), g["noise"])
    torch.manual_seed(SEED)
    n2 = oloop.sample_noise(torch.zeros(4, 128, 6), [True] * 6, angular_var=0.5)
    assert np.array_equal(n2.numpy(), g["noise_var05"])
    torch.manual_seed(SEED)  # RNG anchor of SURVEY.md A.3
    assert torch.allclose(torch.randn(4, 64, 6)[0, 0, :3], torch.tensor([1.5592289, -0.6022594, -1.6624004]), atol=1e-6)


def test_forward_golden_mini(mini_oracle):
    model, sd, cfg = mini_oracle
    g = load_golden("mini_forward.npz")
    x, t = torch.from_numpy(g["x"]), torch.from_numpy(g["t"])
    lengths = g["lengths"].tolist()
    mask = torch.zeros(x.shape[:2])
    for i, n in enumerate(lengths):
        mask[i, :n] = 1.0
    eps = model(x, t, attention_mask=mask)
    assert torch.allclose(eps, torch.from_numpy(g["eps_f32"]), atol=2e-6, rtol=0)
    # values printed in SURVEY.md A.4 by an independent restatement
    assert torch.allclose(eps[0, 0], torch.tensor([-0.236041, -0.427451, 0.182558, -0.877151, 0.052162, 0.688431]), atol=2e-6)
    assert torch.allclose(eps[2, 32], torch.tensor([-1.817486, -0.752683, -0.786334, -0.522085, -0.750055, -0.063359]), atol=2e-6)
    valid = mask.bool()
    assert abs(float(eps[valid].sum()) - (-82.188598)) < 1e-3
    assert abs(float(eps[valid].abs().sum()) - 976.423193) < 1e-2
    # fp32 vs fp64 restatement: the fp32 arithmetic floor
    assert float((eps.double() - torch.from_numpy(g["eps_f64"]))[valid].abs().max()) < 2e-5


def test_forward_properties(mini_oracle):
    """The properties the reference pins in tests/test_transformer.py:83-162, on the oracle."""
    model, _, _ = mini_oracle
    g = torch.Generator().manual_seed(6489)
    x = torch.randn(5, 48, 6, generator=g)
    t = torch.randint(0, 250, (5,), generator=g)
    lengths = [48, 40, 17, 48, 31]
    mask = torch.zeros(5, 48)
    for i, n in enumerate(lengths):
        mask[i, :n] = 1.0
    a = model(x, t, attention_mask=mask)
    assert torch.equal(a, model(x, t, attention_mask=mask))  # determinism
    x2 = x.clone()
    x2[mask == 0] += torch.randn(int((mask == 0).sum()), 6, generator=g)  # noise on masked residues
    b = model(x2, t, attention_mask=mask)
    assert torch.allclose(a[mask.bool()], b[mask.bool()], rtol=1e-3, atol=1e-6)  # mask invariance
    perm = torch.tensor([3, 0, 4, 1, 2])
    c = model(x[perm], t[perm], attention_mask=mask[perm])
    assert torch.allclose(a[perm][mask[perm].bool()], c[mask[perm].bool()], atol=1e-5)  # batch order


def test_chain_golden(mini_oracle):
    model, _, _ = mini_oracle
    g = load_golden("mini_chain.npz")
    # one reference p_sample step (SURVEY.md A.4)
    x = torch.from_numpy(g["step_x"])
    betas = osched.betas_for("cosine", 250)
    torch.manual_seed(SEED)
    y = oloop.p_sample(model, x, torch.full((4,), 100), g["step_lengths"].tolist(), betas)
    assert torch.allclose(y, torch.from_numpy(g["step_y"]), atol=2e-6)
    assert torch.allclose(y[0, 0], torch.tensor([0.037763, -0.548581, 0.003287, -0.841776, 0.140185, 0.678892]), atol=2e-6)
    # short chain, last 12 steps of the linear schedule (cheap) re-run from the golden history
    hist = torch.from_numpy(g["linear100_hist"])
    lens = g["linear100_lengths"].tolist()
    betas = osched.betas_for("linear", 100)
    start = hist[100 - 12 - 1]
    torch.manual_seed(3)
    z = [torch.randn(4, 64, 6) for _ in range(12)]
    out = oloop.p_sample_loop(model, lens, start, 100, betas, [True] * 6, z_list=z, start_t=12)
    assert out.shape == (12, 4, 64, 6)
    assert float(out.abs().max()) <= np.pi + 1e-6


LIVE_T, LIVE_LENGTHS = 20, [40, 33, 40]


def live_noise():
    torch.manual_seed(11)
    return oloop.sample_noise(torch.zeros(3, 40, 6), [True] * 6)


def test_oracle_loop_equals_reference_loop_live(mini_oracle):
    """
    The reference's own loop vs the restated loop, bit for bit.  tests/golden/ref_loop.npz holds the digest of the
    stock p_sample_loop run around this oracle forward (tests/golden/make_golden_reference.py) and every call it made to
    the model; the restated loop is handed the same predictions (oracle/replay.py), and the forward is checked against
    them.
    """
    model, _, _ = mini_oracle
    g = load_golden("ref_loop.npz")
    betas = osched.betas_for("cosine", LIVE_T)
    assert digest(betas) == str(g["loop_betas"])
    noise = live_noise()
    replay = Replay(g, "loop")
    torch.manual_seed(12)
    b = oloop.p_sample_loop(replay, LIVE_LENGTHS, noise, LIVE_T, betas, [True] * 6)
    assert replay.calls == replay.total == LIVE_T
    assert digest(b) == str(g["loop_hist"])
    assert digest(oloop.wrap(noise * 3)) == str(g["loop_wrap3"])
    mask = torch.zeros(3, 40)
    for i, n in enumerate(LIVE_LENGTHS):
        mask[i, :n] = 1.0
    for k in range(LIVE_T):  # the predictions replayed above are this forward's, to the fp32 floor of another CPU
        x = noise if k == 0 else b[k - 1]
        eps = model(x, torch.full((3,), LIVE_T - 1 - k), attention_mask=mask)
        assert torch.allclose(eps, torch.from_numpy(g[f"loop_eps_{k}"]), atol=2e-6, rtol=0)
