"""-m gpu: mask priors and mean-field sampling kernels (SURVEY.md 8f N2/N3) against the oracle and the committed
reference fixtures, forward and backward, through the reference-named helpers."""
import pytest
import torch

from oracle import parts as OPARTS
from oracle import priors as OR
from util import assert_bitexact, assert_close, own_error_atol

pytestmark = pytest.mark.gpu

SHAPES = [(2, 8, 8, 4), (1, 6, 10, 25), (3, 64, 64, 16), (4, 128, 128, 16), (2, 96, 80, 32), (70, 16, 16, 8),
          (1, 1, 9, 4), (1, 9, 1, 3)]


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


def _probs(B, H, W, K, seed):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, H, W, K, generator=g)
    return logits, torch.softmax(logits, dim=-1), g


@pytest.mark.parametrize("B,H,W,K", SHAPES)
def test_mumford_shah(ups, B, H, W, K):
    _, p, g = _probs(B, H, W, K, seed=B * 7 + K)
    alpha = 1.5
    lam = float(alpha * OR.tf_squared_grad(p).median())          # both branches of the minimum occur
    p_o = p.clone().requires_grad_(True)
    outs_o = OR.mumford_shah(p_o, alpha, lam)
    assert 0.2 < float((outs_o[1] > 0).float().mean()) < 0.8
    p_c = p.cuda().requires_grad_(True)
    outs = ups.nn.mumford_shah(p_c, alpha, lam)
    for got, want, name in zip(outs, outs_o, ("r", "smoothness_cost", "contour_cost")):
        assert_bitexact(got, want.detach(), name)
    assert_bitexact(ups.nn.edge_set(p_c, alpha, lam), OR.edge_set(p, alpha, lam), "edge_set")
    cots = [torch.randn(p.shape, generator=g) for _ in range(3)]
    (d_o,) = torch.autograd.grad(outs_o, [p_o], cots)
    (d,) = torch.autograd.grad(outs, [p_c], [c.cuda() for c in cots])
    assert_close(d, d_o, "d x (elementwise cotangents)")
    # only one output used
    (d1_o,) = torch.autograd.grad(OR.mumford_shah(p_o, alpha, lam)[2], p_o, cots[2])
    (d1,) = torch.autograd.grad(ups.nn.mumford_shah(p_c, alpha, lam)[2], p_c, cots[2].cuda())
    assert_close(d1, d1_o, "d x (contour only)")


@pytest.mark.parametrize("B,H,W,K", SHAPES)
def test_mumford_shah_sums(ups, B, H, W, K):
    """The form the training step uses (cub/code/SB_model48i/model.py:744-769): squared spatial sums."""
    _, p, g = _probs(B, H, W, K, seed=B * 11 + K)
    alpha = 1.0
    lam = float(alpha * OR.tf_squared_grad(p).median())
    p_o = p.clone().requires_grad_(True)
    s_o = OR.mumford_shah_sums(p_o, alpha, lam)
    p_c = p.cuda().requires_grad_(True)
    s = ups.nn.mumford_shah_sums(p_c, alpha, lam)
    assert tuple(s.shape) == (B, 4, K)
    # the kernel sums the fp32 maps, which are the oracle's bit for bit: their float64 sum is the exact value
    s64 = torch.stack([v.double().sum(dim=(1, 2)) for v in (*OR.mumford_shah(p, alpha, lam), p)], dim=1)
    for i, name in enumerate(("r", "smoothness_cost", "contour_cost", "x")):
        assert_close(s[:, i], s64[:, i], f"sum {name}", atol=own_error_atol(s_o[:, i], s64[:, i]))
    gs = torch.randn(B, 4, K, generator=g)
    (d_o,) = torch.autograd.grad(s_o, p_o, gs)
    (d,) = torch.autograd.grad(s, p_c, gs.cuda())
    assert_close(d, d_o, "d x (sum cotangents)")
    # the reference's loss: mean_b sum_k (sum_hw .)^2 for each of the four maps
    loss_o = (OR.mumford_shah_sums(p_o, alpha, lam) ** 2).sum(dim=2).mean(dim=0).sum()
    loss = (ups.nn.mumford_shah_sums(p_c, alpha, lam) ** 2).sum(dim=2).mean(dim=0).sum()
    assert_close(loss, loss_o.detach(), "squared-sum loss", rtol=1e-4, atol=1e-5 * float(loss_o.detach().abs()))
    (dl_o,) = torch.autograd.grad(loss_o, p_o)
    (dl,) = torch.autograd.grad(loss, p_c)
    assert_close(dl, dl_o, "d loss", atol=1e-5 * float(dl_o.abs().max().clamp(min=1.0)))


@pytest.mark.parametrize("B,H,W,K", SHAPES)
def test_logit_priors(ups, B, H, W, K):
    logits, _, g = _probs(B, H, W, K, seed=B * 13 + K)
    x_o = logits.clone().requires_grad_(True)
    pri_o = OR.logit_priors(x_o)
    x_c = logits.cuda().requires_grad_(True)
    dist = ups.nn.MeanFieldDistribution(x_c, K)
    pri = torch.stack([dist.kl(), dist.kl_improper_gmrf(), dist.kl_tv()])
    assert_close(pri, pri_o.detach(), "kl / gmrf / tv")
    cot = torch.randn(3, generator=g) * B                        # keeps the gradient entries O(1)
    (d_o,) = torch.autograd.grad(pri_o, x_o, cot)
    (d,) = torch.autograd.grad(pri, x_c, cot.cuda())
    assert_close(d, d_o, "d logits")
    for i in range(3):                                           # each energy on its own
        (di_o,) = torch.autograd.grad(OR.logit_priors(x_o)[i], x_o, torch.tensor(float(B)))
        (di,) = torch.autograd.grad(ups.nn.MeanFieldDistribution(x_c, K)._all()[i], x_c, torch.tensor(float(B)).cuda())
        assert_close(di, di_o, f"d logits (energy {i})")


@pytest.mark.parametrize("B,H,W,K", SHAPES)
@pytest.mark.parametrize("noise", [1.0, 0.7])
def test_mean_field_sample_and_fused_softmax(ups, B, H, W, K, noise):
    logits, _, g = _probs(B, H, W, K, seed=B * 17 + K)
    eps = torch.randn(B, H, W, K, generator=g)
    want = OR.mean_field_sample(logits, eps, noise)
    x_c = logits.cuda().requires_grad_(True)
    dist = ups.nn.MeanFieldDistribution(x_c, K)
    got = dist.sample(noise, eps=eps.cuda())
    assert_bitexact(got, want, "sample")
    # fused sample + softmax + labels + straight-through mask == the chain of the stand-alone pieces
    p_o = OPARTS.softmax(want)
    hard_o = OPARTS.straight_through_estimator(OPARTS.hard_max(p_o, 3), p_o)
    l, p, labels, hard = dist.sample_softmax(noise, eps=eps.cuda())
    assert_bitexact(l, want, "sampled logits")
    assert_bitexact(p, p_o, "probs")
    assert_bitexact(hard, hard_o, "hard mask")
    assert labels.dtype == torch.int64 and torch.equal(labels.cpu(), OPARTS.argmax_labels(p_o))
    # gradient: identity through the sample, softmax-bwd through probs + hard (straight-through)
    g_p, g_h, g_l = (torch.randn(B, H, W, K, generator=g) for _ in range(3))
    x_o = logits.clone().requires_grad_(True)
    s_o = OR.mean_field_sample(x_o, eps, noise)
    pp = OPARTS.softmax(s_o)
    hh = OPARTS.straight_through_estimator(OPARTS.hard_max(pp, 3), pp)
    (d_o,) = torch.autograd.grad([pp, hh, s_o], [x_o], [g_p, g_h, g_l])
    (d,) = torch.autograd.grad([p, hard, l], [x_c], [g_p.cuda(), g_h.cuda(), g_l.cuda()])
    assert_close(d, d_o, "d mean")
    # non-stochastic distribution returns the mean itself (nn.py:1422-1423)
    assert ups.nn.MeanFieldDistribution(x_c, K, stochastic=False).sample() is x_c


@pytest.mark.parametrize("B,H,W,K", SHAPES)
@pytest.mark.parametrize("entropy_func", ["cross_entropy", "entropy"])
def test_weak_cross_entropy(ups, B, H, W, K, entropy_func):
    logits, _, g = _probs(B, H, W, K, seed=B * 19 + K)
    logits = logits * 2
    logits[0, 0] = torch.round(logits[0, 0])                     # exact ties: hard_max marks every maximum
    x_o = logits.clone().requires_grad_(True)
    v_o = OR.weak_cross_entropy(x_o, entropy_func)
    x_c = logits.cuda().requires_grad_(True)
    v = ups.model.weak_cross_entropy(x_c, entropy_func)
    assert_close(v, v_o.detach(), entropy_func)
    cot = 0.9 * B * H * W
    (d_o,) = torch.autograd.grad(v_o, x_o, torch.tensor(cot))
    (d,) = torch.autograd.grad(v, x_c, torch.tensor(cot).cuda())
    assert_close(d, d_o, f"d logits ({entropy_func})")


def test_weak_cross_entropy_rejects_unknown_mode(ups):
    with pytest.raises(ValueError):
        ups.model.weak_cross_entropy(torch.zeros(1, 2, 2, 4).cuda(), "nope")


@pytest.mark.parametrize("B,H,W,K", SHAPES)
def test_mask2rgb(ups, B, H, W, K):
    _, p, g = _probs(B, H, W, K, seed=B * 23 + K)
    p[0, 0, :, :] = 0.25                                          # ties -> first maximum
    colors = torch.rand(K, 3, generator=g)
    assert_close(ups.nn.mask2rgb(p.cuda(), True, colors=colors), OR.mask2rgb(p, colors, True), "hot", rtol=0, atol=0)
    assert_close(ups.nn.mask2rgb(p.cuda(), False, colors=colors), OR.mask2rgb(p, colors, False), "soft")
    assert tuple(ups.nn.mask2rgb(p.cuda()).shape) == (B, H, W, 3)


def test_priors_reference_fixture(ups, golden):
    """The kernels against what the reference's own function bodies produced (tests/golden/priors.npz)."""
    g = golden("priors.npz")
    t = lambda k: torch.from_numpy(g[k])                          # noqa: E731
    for tag in ("a", "b"):
        alpha, lam = float(g[f"{tag}_alpha"]), float(g[f"{tag}_lam"])
        p = t(f"{tag}_p").cuda().requires_grad_(True)
        outs = ups.nn.mumford_shah(p, alpha, lam)
        for got, k in zip(outs, ("r", "smooth", "contour")):
            assert_bitexact(got, t(f"{tag}_{k}"), f"{tag} {k}")
        assert_bitexact(ups.nn.edge_set(p, alpha, lam), t(f"{tag}_edges"), f"{tag} edges")
        (d,) = torch.autograd.grad(outs, [p], [t(f"{tag}_g_{k}").cuda() for k in ("r", "smooth", "contour")])
        assert_close(d, t(f"{tag}_d_p_elem"), f"{tag} d p (elementwise)")
        sums = ups.nn.mumford_shah_sums(p, alpha, lam)
        for i, k in enumerate(("sum_r", "sum_smooth", "sum_contour", "sum_p")):
            assert_close(sums[:, i], t(f"{tag}_{k}"), f"{tag} {k}")
        gs = torch.stack([t(f"{tag}_g_{k}") for k in ("sum_r", "sum_smooth", "sum_contour", "sum_p")], dim=1).cuda()
        (d,) = torch.autograd.grad(sums, p, gs)
        assert_close(d, t(f"{tag}_d_p_sums"), f"{tag} d p (sums)")

        logits = t(f"{tag}_logits").cuda().requires_grad_(True)
        K = logits.shape[-1]
        dist = ups.nn.MeanFieldDistribution(logits, K)
        assert_bitexact(dist.sample(0.7, eps=t(f"{tag}_eps").cuda()), t(f"{tag}_sample"), f"{tag} sample")
        for fn, k in ((dist.kl, "kl0"), (dist.kl_improper_gmrf, "gmrf"), (dist.kl_tv, "tv")):
            assert_close(fn(), t(f"{tag}_{k}"), f"{tag} {k}")
        (d,) = torch.autograd.grad(dist.kl_improper_gmrf(), logits, retain_graph=True)
        assert_close(d, t(f"{tag}_d_gmrf"), f"{tag} d gmrf")
        (d,) = torch.autograd.grad(dist.kl(), logits)
        assert_close(d, t(f"{tag}_d_kl0"), f"{tag} d kl0")
        for mode, k in (("cross_entropy", "ce"), ("entropy", "ent")):
            v = ups.model.weak_cross_entropy(logits, mode)
            assert_close(v, t(f"{tag}_{k}"), f"{tag} {k}")
            (d,) = torch.autograd.grad(v, logits)
            assert_close(d, t(f"{tag}_d_{k}"), f"{tag} d {k}")
        colors = t(f"{tag}_colors")
        assert_close(ups.nn.mask2rgb(p, True, colors=colors), t(f"{tag}_rgb_hot"), f"{tag} rgb hot", rtol=0, atol=0)
        assert_close(ups.nn.mask2rgb(p, False, colors=colors), t(f"{tag}_rgb_soft"), f"{tag} rgb soft")


def test_known_answers(ups):
    """A constant map has zero finite-difference energy except at the right / bottom border, where the zero padding
    of the SAME convolution makes gx / gy = 0.25*x; a vertical step edge is found by edge_set."""
    x = torch.full((1, 6, 6, 4), 0.8)
    r, smooth, contour = ups.nn.mumford_shah(x.cuda(), 1.0, 1e-2)
    assert float(r[0, :5, :5].abs().max()) == 0.0
    assert_close(r[0, 2, 5], torch.full((4,), 1e-2), "border clamps to lambda")          # (0.25*0.8)^2 = 0.04 > lambda
    assert_close(contour[0, 5, 5], torch.full((4,), 1e-2), "corner")
    assert float(smooth[0, 2, 5].abs().max()) == 0.0
    step = torch.zeros(1, 6, 6, 4)
    step[:, :, 3:] = 1.0
    e = ups.nn.edge_set(step.cuda(), 1.0, 1e-2)
    assert e[0, :5, 2].min() == 1.0 and e[0, :5, :2].max() == 0.0
    const = ups.nn.MeanFieldDistribution(torch.full((2, 5, 5, 4), 3.0).cuda(), 4)
    assert float(const.kl_improper_gmrf()) == 0.0 and float(const.kl_tv()) == 0.0
    assert_close(const.kl(), torch.tensor(0.5 * 9.0 * 100), "kl of a constant")
