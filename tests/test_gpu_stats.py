"""-m gpu: mask-statistics kernels (SURVEY.md 8f N1/N2) against the oracle and the committed
reference fixtures, forward and backward, through the reference-named helpers."""
import numpy as np
import pytest
import torch

from oracle import stats as OS
from util import assert_close, own_error_atol

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


def _density(B, H, W, K, seed):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, H, W, K, generator=g) * 3
    dens = torch.softmax(logits.reshape(B, H * W, K), dim=1).reshape(B, H, W, K)   # sums to 1 over HW
    sf = torch.rand(B, K, generator=g) * 0.5 + 0.75
    return logits, dens, sf, g


@pytest.mark.parametrize("B,H,W,K", [(2, 8, 8, 4), (1, 6, 10, 25), (3, 64, 64, 16), (8, 128, 128, 16), (2, 96, 80, 32),
                                     (70, 32, 32, 8)])
def test_probs_to_mu_sigma(ups, B, H, W, K):
    _, dens, sf, g = _density(B, H, W, K, seed=B + K)
    d_o = dens.clone().requires_grad_(True)
    mu_o, sigma_o = OS.probs_to_mu_sigma(d_o, sf)
    g_mu, g_sigma = torch.randn(mu_o.shape, generator=g), torch.randn(sigma_o.shape, generator=g)
    (dd_o,) = torch.autograd.grad([mu_o, sigma_o], [d_o], [g_mu, g_sigma])
    d_c = dens.cuda().requires_grad_(True)
    mu, sigma = ups.nn.probs_to_mu_sigma(d_c, sf.cuda())
    assert tuple(mu.shape) == (B, K, 2) and tuple(sigma.shape) == (B, K, 2, 2)
    # sums of H*W terms: against the same expression in float64, within the fp32 oracle's own error
    mu64, sigma64 = OS.probs_to_mu_sigma(dens.double(), sf.double())
    assert_close(mu, mu64, "mu", atol=own_error_atol(mu_o, mu64))
    assert_close(sigma, sigma64, "sigma", atol=own_error_atol(sigma_o, sigma64))
    (dd,) = torch.autograd.grad([mu, sigma], [d_c], [g_mu.cuda(), g_sigma.cuda()])
    assert_close(dd, dd_o, "d probs")
    # only one of the two outputs used
    (dd2,) = torch.autograd.grad(ups.nn.probs_to_mu_sigma(d_c, sf.cuda())[0].sum(), d_c)
    (dd2_o,) = torch.autograd.grad(OS.probs_to_mu_sigma(d_o, sf)[0].sum(), d_o)
    assert_close(dd2, dd2_o, "d probs (mu only)")


def test_probs_to_mu_sigma_reference_fixture(ups, golden):
    g = golden("stats.npz")
    for tag in ("a", "b"):
        dens = torch.from_numpy(g[f"{tag}_dens"]).cuda().requires_grad_(True)
        mu, sigma = ups.nn.probs_to_mu_sigma(dens, torch.from_numpy(g[f"{tag}_sf"]).cuda())
        assert_close(mu, torch.from_numpy(g[f"{tag}_mu"]), f"{tag} mu")
        assert_close(sigma, torch.from_numpy(g[f"{tag}_sigma"]), f"{tag} sigma")
        (d,) = torch.autograd.grad([mu, sigma], [dens], [torch.from_numpy(g[f"{tag}_g_mu"]).cuda(),
                                                         torch.from_numpy(g[f"{tag}_g_sigma"]).cuda()])
        assert_close(d, torch.from_numpy(g[f"{tag}_d_dens"]), f"{tag} d dens")
        p = torch.from_numpy(g[f"{tag}_p"]).cuda().requires_grad_(True)
        kl = ups.model.categorical_kl(p)
        assert_close(kl, torch.from_numpy(g[f"{tag}_kl"]), f"{tag} kl")
        (dp,) = torch.autograd.grad(kl, p)
        assert_close(dp, torch.from_numpy(g[f"{tag}_d_p"]), f"{tag} d p")


def test_known_answers(ups):
    """A delta density at pixel (i, j) has mu = grid(i, j) and zero covariance; a uniform
    density has mu = 0; uniform probabilities have zero categorical KL."""
    B, H, W, K = 1, 16, 16, 4
    dens = torch.zeros(B, H, W, K)
    dens[0, 3, 12, 0] = 1.0
    dens[0, :, :, 1] = 1.0 / (H * W)
    mu, sigma = ups.nn.probs_to_mu_sigma(dens.cuda(), torch.ones(B, K).cuda())
    lin = torch.linspace(-1, 1, H)
    assert_close(mu[0, 0], torch.stack([lin[3], lin[12]]), "delta mu")
    assert_close(sigma[0, 0], torch.zeros(2, 2), "delta sigma", atol=1e-6)
    assert_close(mu[0, 1], torch.zeros(2), "uniform mu", atol=1e-6)
    assert float(ups.model.categorical_kl(torch.full((2, 8, 8, 16), 1 / 16.0).cuda()).abs()) < 1e-6


@pytest.mark.parametrize("shape", [(2, 8, 8, 4), (1, 7, 9, 25), (8, 128, 128, 16), (3, 5, 5, 3)])
def test_categorical_kl(ups, shape):
    g = torch.Generator().manual_seed(sum(shape))
    p = torch.softmax(torch.randn(*shape, generator=g) * 2, dim=-1)
    p_o = p.clone().requires_grad_(True)
    kl_o = OS.categorical_kl(p_o)
    n_pix = p.numel() // p.shape[-1]
    cot = 0.7 * n_pix                                    # keeps the gradient entries O(1)
    (dp_o,) = torch.autograd.grad(kl_o, p_o, torch.tensor(cot))
    p_c = p.cuda().requires_grad_(True)
    kl = ups.model.categorical_kl(p_c)
    assert_close(kl, kl_o.detach(), "kl")
    (dp,) = torch.autograd.grad(kl, p_c, torch.tensor(cot).cuda())
    assert_close(dp, dp_o, "d kl")


def test_draw_rect_and_patch_masks(ups=None):
    """SURVEY.md 8f N1: tfutils.draw_rect / the patch masks of model.py:437-445 (source un-vendored: the oracle restates
    the library's documented convention; borders, zero-size and out-of-image centres included)."""
    import ups_b200
    from oracle import parts as OP
    from oracle import stats as OS_
    centers = torch.tensor([[0, 0], [5, 7], [15, 15], [-3, 4], [20, 2], [8, 8]], dtype=torch.int32)
    for ph, pw in ((5, 5), (4, 6), (1, 1), (0, 3), (40, 40)):
        got = ups_b200.nn.draw_rect(centers.cuda(), ph, pw, [16, 12, 1])
        assert got.shape == (6, 16, 12, 1)
        assert torch.equal(got[..., 0].cpu(), OS_.draw_rect(centers, ph, pw, 16, 12)), (ph, pw)
    g = torch.Generator().manual_seed(0)
    p = OP.softmax(torch.randn(3, 24, 24, 16, generator=g))
    mh = OP.straight_through_estimator(OP.hard_max(p, 3), p)
    got = ups_b200.nn.patch_masks(mh.cuda(), 7, gamma=3.0)
    want = OS_.patch_masks(mh, 7, gamma=3.0)
    assert got.shape == (3, 24, 24, 16)
    # the centre of mass is a float reduction: a centre within rounding of an integer boundary may land one pixel off
    same = (got.cpu() == want).all(1).all(1)          # [N, K]
    assert same.float().mean() >= 0.9, same
    assert torch.equal(got.cpu().sum((1, 2))[same], want.sum((1, 2))[same])
