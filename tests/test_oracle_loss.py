"""
SURVEY.md section 8f rank 3 (training step) - groundwork on the CPU: the restated objective `oracle/loss.py` pinned
(1) on the known answers the reference's own tests hold (/root/reference/tests/test_losses.py:10-160 and the doctests of
    /root/reference/foldingdiff/losses.py:15-19, :43-44),
(2) BIT-identically against what the stock package computed on the same inputs: `foldingdiff.losses` and the
    unmodified `BertForDiffusion._get_loss_terms` (modelling.py:553-604) driven with a stand-in `self`,
(3) its closed-form gradient against torch autograd through the reference's own functions.
No CUDA kernel for this row exists yet (DESIGN.md section 0, row f); nothing here touches the product path.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import loss as oloss

IS_ANGULAR = [False, True, True, True]  # one non-angular feature, then angles (the default `is_angle` of p_sample_loop, sampling.py:84)
IS_ANGULAR6 = [True] * 6                 # canonical-full-angles: every feature is an angle


def t(x, dtype=torch.float32):
    return torch.tensor(x, dtype=dtype)


# ---- (1) the reference's own known answers ---------------------------------------------------------------------------

@pytest.mark.parametrize("pred, target, beta, want, places", [
    (0.1, 2 * np.pi, 1.0, 0.0050, 6),            # test_easy
    (0.1, 2 * np.pi - 0.1, 1.0, 0.02, 6),        # test_rounding
    (0.0, 3.14, 1.0, 2.64, 5),                   # test_no_rounding
    (2.0, 4.0, 1.0, 1.5, 5),                     # test_double_positive_rounding
    (-0.1, np.pi + 2, 0.1, 0.991593, 5),         # test_neg_pos
    (0.5, -np.pi, 0.1, 2.591593, 5),             # test_neg_pos_2
    (-17.0466, -1.3888, 0.1, 3.0414, 4),         # doctest losses.py:43-44
])
def test_smooth_l1_known_answers_of_the_reference_tests(pred, target, beta, want, places):
    got = oloss.radian_smooth_l1(t(pred), t(target), beta=beta).item()
    assert abs(got - want) < 0.5 * 10 ** (-places) + 1e-7, (got, want)


def test_smooth_l1_is_periodic_in_both_arguments_and_symmetric():
    # test_zeros, test_loop_* and test_symmetric of the reference's test_losses.py
    for i in range(-10, 10):
        assert abs(oloss.radian_smooth_l1(t(0.0), t(i * 2 * np.pi)).item()) < 1e-5
    for x, y, want in [(-0.1, -1.0, 0.85), (-0.1, 1.0, 1.05), (0.1, -1.0, 1.05), (0.1, 1.0, 0.85)]:
        for i in range(-10, 10):
            for j in range(-10, 10):
                got = oloss.radian_smooth_l1(t(x + i * 2 * np.pi), t(y + j * 2 * np.pi), beta=0.1).item()
                assert abs(got - want) < 5e-5, (x, y, i, j, got)
    rng = np.random.default_rng(6489)
    for _ in range(100):
        x, y = rng.uniform(low=-200 * np.pi, high=200 * np.pi, size=2)
        a = oloss.radian_smooth_l1(t(x, torch.float64), t(y, torch.float64)).item()
        b = oloss.radian_smooth_l1(t(y, torch.float64), t(x, torch.float64)).item()
        assert abs(a - b) < 1e-7


def test_l1_known_answers_of_the_reference_doctests():
    assert abs(oloss.radian_l1(t(0.1), t(2 * np.pi)).item() - 0.1) < 1e-6
    assert abs(oloss.radian_l1(t(0.1), t(2 * np.pi - 0.1)).item() - 0.2) < 1e-6


# ---- synthetic training batch ----------------------------------------------------------------------------------------

def _batch(seed=0, B=7, N=24, F=6, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    lengths = torch.randint(5, N + 1, (B,), generator=g)
    lengths[0] = N
    mask = (torch.arange(N)[None, :] < lengths[:, None]).to(torch.float32)
    known = torch.randn(B, N, F, generator=g)
    pred = known + scale * torch.randn(B, N, F, generator=g)  # differences on both sides of beta and beyond +-pi
    return pred, known, mask


def test_terms_ignore_padded_positions_and_average_over_valid_tokens():
    pred, known, mask = _batch()
    a = oloss.loss_terms(pred, known, mask, IS_ANGULAR6)
    junk = pred.clone()
    junk[mask == 0] = 1e6
    assert torch.equal(a, oloss.loss_terms(junk, known, mask, IS_ANGULAR6))
    # per-feature value == plain mean over the valid elements of the elementwise Huber
    d = oloss.wrap(known - pred, -torch.pi, torch.pi)
    h = torch.where(d.abs() < oloss.ANGULAR_BETA, 0.5 * d ** 2 / oloss.ANGULAR_BETA, d.abs() - 0.5 * oloss.ANGULAR_BETA)
    want = (h * mask[..., None]).sum((0, 1)).double() / mask.sum().double()
    assert torch.allclose(a.double(), want, rtol=1e-6, atol=1e-7)


def test_uninformed_predictor_anchor():
    # a predictor that returns 0 against standard-normal angular noise: the level a fresh model starts from
    g = torch.Generator().manual_seed(3)
    known = torch.randn(64, 128, 6, generator=g)
    mask = torch.ones(64, 128)
    got = oloss.training_loss(torch.zeros_like(known), known, mask, IS_ANGULAR6).item()
    assert abs(got - oloss.expected_loss_of_uninformed_predictor()) < 0.01
    assert 0.55 < got < 0.75


# ---- (2) + (3): against the stock reference ------------------------------------------------------------------------
# tests/golden/ref_loss.npz holds what the stock package (baseline/_ref) computed on these inputs: written by
# tests/golden/make_golden_reference.py, which drives the unmodified `_get_loss_terms` with a stand-in `self`.

LOSS_FN_SHAPES = [(), (1,), (977,), (33, 7)]
BETAS = (1.0, 0.1, float(torch.pi / 10))
CIRCLE_PENALTIES = (0.0, 0.3)
TERMS_FEATURES = [IS_ANGULAR6, IS_ANGULAR, [False, False, True]]
GRAD_FEATURES = [IS_ANGULAR6, IS_ANGULAR]


def loss_fn_inputs():
    g = torch.Generator().manual_seed(11)
    return [(20 * torch.randn(shape, generator=g), 20 * torch.randn(shape, generator=g)) for shape in LOSS_FN_SHAPES]


def features_tag(is_angular):
    return "".join("T" if a else "F" for a in is_angular)


@pytest.fixture(scope="module")
def ref():
    return load_golden("ref_loss.npz")


def test_loss_functions_bit_identical_to_the_reference(ref):
    for i, (x, y) in enumerate(loss_fn_inputs()):
        for b, beta in enumerate(BETAS):
            for c, cp in enumerate(CIRCLE_PENALTIES):
                ours = oloss.radian_smooth_l1(x, y, beta=beta, circle_penalty=cp)
                theirs = torch.from_numpy(ref[f"fn{i}_smooth_l1_{b}_{c}"])
                assert torch.equal(ours, theirs), (x.shape, beta, cp)
        assert torch.equal(oloss.radian_l1(x, y), torch.from_numpy(ref[f"fn{i}_l1"]))


@pytest.mark.parametrize("is_angular", TERMS_FEATURES)
@pytest.mark.parametrize("loss", ["smooth_l1", "l1"])
def test_loss_terms_bit_identical_to_get_loss_terms(ref, is_angular, loss):
    pred, known, mask = _batch(seed=len(is_angular), F=len(is_angular))
    theirs = torch.from_numpy(ref[f"terms_{features_tag(is_angular)}_{loss}"])
    ours = oloss.loss_terms(pred, known, mask, is_angular, loss)
    assert theirs.shape == ours.shape == (len(is_angular),)
    assert torch.equal(ours, theirs)
    assert torch.equal(oloss.training_loss(pred, known, mask, is_angular, loss), torch.mean(theirs))  # modelling.py:685


@pytest.mark.parametrize("is_angular", GRAD_FEATURES)
def test_closed_form_gradient_matches_autograd_through_the_reference(ref, is_angular):
    pred, known, mask = _batch(seed=5, F=len(is_angular))
    theirs = torch.from_numpy(ref[f"grad_{features_tag(is_angular)}"])
    ours = oloss.training_loss_grad(pred.double(), known.double(), mask, is_angular)
    assert torch.all(ours[mask == 0] == 0) and torch.all(theirs[mask == 0] == 0)
    assert torch.allclose(ours, theirs, rtol=1e-12, atol=1e-15)


def test_closed_form_gradient_matches_autograd_through_the_oracle():
    # the same check with autograd through the restatement itself
    for is_angular in (IS_ANGULAR6, IS_ANGULAR):
        pred, known, mask = _batch(seed=9, F=len(is_angular))
        pred = pred.double().requires_grad_(True)
        oloss.training_loss(pred, known.double(), mask, is_angular).backward()
        ours = oloss.training_loss_grad(pred.detach(), known.double(), mask, is_angular)
        assert torch.allclose(ours, pred.grad, rtol=1e-12, atol=1e-15)
