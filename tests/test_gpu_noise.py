"""-m gpu: the mean-field logit noise drawn on the device (PartStep.forward(noise_seed=...), ups_normal_philox_fwd,
ups_part_softmax_sampled_philox_fwd).  The step on means with a seed must equal, bit for bit, today's step fed the logits
l = mean_field_sample(mean, eps, noise_level) with eps = ups_normal_philox_fwd(seed, draw, offset): forward and backward,
in every configuration the step supports."""
import math

import pytest
import torch

from oracle import noise as ON
from oracle import step as OS
from util import assert_bitexact, cuda, make_inputs

pytestmark = pytest.mark.gpu

SEED, LEVEL = 0x5EED_0123_4567_89AB, 0.7


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


def _eps(B, S, K, draw, seed=SEED, offset=0):
    from ups_b200 import ops
    return ops.normal_philox(ops._seed_i64(seed), draw, offset * S * S, B * S * S, K, torch.device("cuda")).view(B, S, S, K)


def _sampled(mean, draw, seed=SEED, level=LEVEL, offset=0):
    from ups_b200 import ops
    B, S, _, K = mean.shape
    return ops.mean_field_sample(mean, _eps(B, S, K, draw, seed, offset), float(level))


def _clone(d):
    return {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in d.items() if v is not None}


def _same(got, want, what, dviews_atol=1e-3):
    assert set(got) == set(want), (what, set(got) ^ set(want))
    for k in want:
        a, b = got[k], want[k]
        if k == "dviews":      # accumulated with atomics (K6): compared as tests/test_gpu_workloads.py does
            assert float((a - b).abs().max()) <= dviews_atol, (what, k)
        elif a.dtype == torch.float32:
            assert_bitexact(a, b, f"{what}: {k}")
        else:
            assert torch.equal(a, b), (what, k)


class Case:
    """One step configuration: inputs on the device, extra forward / backward arguments."""

    def __init__(self, B, S, K, F, V=3, use_tps=True, views_grad=False, first_conv=0, encoder_conv=0, u8=False, seed=3):
        self.B, self.S, self.K, self.F, self.V = B, S, K, F, V
        self.kw = dict(n_views=V, use_tps=use_tps, views_grad=views_grad, first_conv=first_conv, encoder_conv=encoder_conv)
        inp = make_inputs(B, S, K, F, V, seed=seed, ties=True)
        g = torch.Generator().manual_seed(seed + 1)
        self.d = cuda(inp)
        if u8:
            self.d["views"] = ((inp["views"] + 1) * 127.5).round().clamp(0, 255).to(torch.uint8).cuda()
        self.conv = [None] * 4
        c = self.d["cot"]
        self.g1, self.g2 = c["g_inj"], c["g_parts"]
        if first_conv:
            sd = math.sqrt(1.0 / ((F + K) * 9))
            self.conv[0] = ((torch.rand(3, 3, F + K, first_conv, generator=g) * 2 - 1) * sd).cuda()
            self.conv[1] = ((torch.rand(first_conv, generator=g) * 2 - 1) * sd).cuda()
            self.g1 = torch.randn(B, S, S, first_conv, generator=g).cuda()
        if encoder_conv:
            self.conv[2] = (torch.randn(3, 3, 3, encoder_conv, generator=g) * 0.2).cuda()
            self.conv[3] = (torch.randn(encoder_conv, generator=g) * 0.2).cuda()
            self.g2 = torch.randn(K * B, S, S, encoder_conv, generator=g).cuda()
        self.gw = torch.stack(c["g_warped"]).contiguous() if views_grad else None

    def step(self, **kw):
        from ups_b200.step import PartStep
        return PartStep(self.B, self.S, self.K, self.F, **dict(self.kw, **kw))

    def run(self, step, l0, l1, split=False, **noise):
        d = self.d
        if split:
            step.forward_warp(d["views"], d["coord"], d["t_vector"])
            out = step.forward_parts(l0, l1, d["feat"], *self.conv, **noise)
        else:
            out = step.forward(d["views"], d["coord"], d["t_vector"], l0, l1, d["feat"], *self.conv, **noise)
        out = _clone(out)
        c = d["cot"]
        grad = _clone(step.backward(self.g1, self.g2, c["g_pooled"], c["g_m0"], c["g_m1"], self.gw))
        torch.cuda.synchronize()
        return out, grad


def test_normal_philox_equals_oracle(ups):
    from ups_b200 import ops
    for seed, draw, off, n, K in [(0, 0, 0, 100_000, 16), (SEED, 1, 2 ** 32 - 999, 3000, 25), (2 ** 64 - 1, 0, 2 ** 40, 777, 3),
                                  (12, 1, 5, 4096, 32)]:
        got = ops.normal_philox(ops._seed_i64(seed), draw, off, n, K, torch.device("cuda"))
        assert_bitexact(got, ON.normal_philox(seed, draw, off, n, K), f"eps seed={seed} K={K}")


@pytest.mark.parametrize("K", [16, 25, 40])
def test_sampled_softmax_philox_equals_eps_form(ups, K):
    """ups_part_softmax_sampled_philox_fwd (vector and generic kernels) == ups_part_softmax_sampled_fwd fed the draw;
    MeanFieldDistribution.sample / sample_softmax with seed= route to it."""
    from ups_b200 import nn, ops
    g = torch.Generator().manual_seed(K)
    mean = (torch.randn(3, 32, 32, K, generator=g) * 2).cuda()
    mean[:, 0] = torch.round(mean[:, 0])
    eps = _eps(3, 32, K, 1, offset=7)
    want = ops.part_softmax_sampled(mean, eps, LEVEL)
    got = ops.part_softmax_sampled_philox(mean, ops._seed_i64(SEED), 1, 7 * 32 * 32, LEVEL)
    for w, o, name in zip(want, got, ("logits", "probs", "labels", "hard")):
        assert torch.equal(w.view(torch.int32) if w.dtype == torch.float32 else w,
                           o.view(torch.int32) if o.dtype == torch.float32 else o), name
    dist = nn.MeanFieldDistribution(mean, K)
    s = dist.sample(LEVEL, seed=SEED, draw=1, sample_offset=7)
    assert_bitexact(s, want[0], "sample(seed=)")
    ss = dist.sample_softmax(LEVEL, seed=SEED, draw=1, sample_offset=7)
    assert_bitexact(ss[1], want[1], "sample_softmax(seed=) probs")
    m = mean.clone().requires_grad_(True)
    _, p, _, _ = nn.MeanFieldDistribution(m, K).sample_softmax(LEVEL, seed=SEED)
    (dm,) = torch.autograd.grad(p, m, torch.ones_like(p) * torch.arange(K, device="cuda"))
    assert_bitexact(dm, ops.part_softmax_grad(p.detach(), torch.ones_like(p) * torch.arange(K, device="cuda")), "d mean")


CONFIGS = {
    "fused": dict(B=4, S=64, K=16, F=64),
    "fused_views_grad": dict(B=3, S=64, K=16, F=32, views_grad=True),
    "two_launches": dict(B=3, S=64, K=32, F=64, split=True),
    "padded_k25": dict(B=3, S=64, K=25, F=64),
    "padded_k25_pitched": dict(B=3, S=64, K=25, F=64, pitched=True),
    "padded_k12_two_views": dict(B=2, S=32, K=12, F=16, V=2),
    "first_conv": dict(B=2, S=64, K=16, F=64, first_conv=32),
    "first_conv_k25_generic": dict(B=2, S=32, K=25, F=16, first_conv=16),
    "both_convs": dict(B=2, S=32, K=8, F=16, first_conv=16, encoder_conv=8),
    "generic_f10": dict(B=2, S=32, K=16, F=10),
    "generic_k40": dict(B=1, S=32, K=40, F=16),
    "no_tps": dict(B=3, S=64, K=16, F=64, V=2, use_tps=False),
    "uint8_views": dict(B=2, S=64, K=16, F=64, u8=True),
    "sample_offset": dict(B=2, S=64, K=16, F=64, offset=37),
    "cub_b256_k16": dict(B=256, S=128, K=16, F=64),
    "cub_b256_k25": dict(B=256, S=128, K=25, F=64),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_step_with_seed_equals_step_on_sampled_logits(ups, name):
    from ups_b200 import _cabi as C
    cfg = dict(CONFIGS[name])
    split, pitched, offset = cfg.pop("split", False), cfg.pop("pitched", False), cfg.pop("offset", 0)
    case = Case(**cfg)
    d = case.d
    ref = case.step(sample_offset=offset)
    want = case.run(ref, _sampled(d["l0"], 0, offset=offset), _sampled(d["l1"], 1, offset=offset), split=split)
    C.launch_count_reset()
    case.run(ref, d["l0"], d["l1"], split=split)
    n_plain = C.launch_count()
    step = case.step(sample_offset=offset)
    l0, l1 = d["l0"], d["l1"]
    if pitched:
        pi = step.pitched_inputs()
        pi["l0"].copy_(l0)
        pi["l1"].copy_(l1)
        l0, l1 = pi["l0"], pi["l1"]
    C.launch_count_reset()
    got = case.run(step, l0, l1, split=split, noise_seed=SEED, noise_level=LEVEL)
    assert C.launch_count() == n_plain, "the draw adds no launch"
    _same(got[0], want[0], f"{name} forward")
    _same(got[1], want[1], f"{name} backward")


def test_seeded_step_against_chained_oracle_cub_b8(ups):
    """B=8 CUB slice with a seed against the chained oracle (oracle/noise.py), at the bar of test_gpu_step:
    warped views, probabilities, labels and part images bit for bit."""
    from test_gpu_step import _check
    from ups_b200.step import PartStep
    B, S, K, F, V = 8, 128, 16, 64, 3
    inp = make_inputs(B, S, K, F, V, seed=21, ties=True)
    cot = dict(inp["cot"], g_warped=None)
    out_o, grad_o = ON.step_forward_backward([v for v in inp["views"]], inp["coord"], inp["t_vector"], inp["l0"], inp["l1"],
                                             inp["feat"], cot, SEED, noise_level=LEVEL, sample_offset=3)
    grad_o["_ref64"] = OS.reduction_refs_fp64([v for v in inp["views"]], inp["coord"], inp["t_vector"], out_o, cot)
    step = PartStep(B, S, K, F, n_views=V, sample_offset=3)
    d = cuda(inp)
    out = step.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"], noise_seed=SEED, noise_level=LEVEL)
    grad = step.backward(d["cot"]["g_inj"], d["cot"]["g_parts"], d["cot"]["g_pooled"], d["cot"]["g_m0"], d["cot"]["g_m1"])
    torch.cuda.synchronize()
    _check(out, grad, out_o, grad_o)
    # the noise moved the labels (the seed reached the kernels)
    assert not torch.equal(out_o["labels0"], OS.step_forward([v for v in inp["views"]], inp["coord"], inp["t_vector"],
                                                             inp["l0"], inp["l1"], inp["feat"])["labels0"])


@pytest.mark.parametrize("name", ["fused", "padded_k25", "generic_f10", "first_conv"])
def test_zero_noise_level_equals_noise_free_step(ups, name):
    cfg = dict(CONFIGS[name])
    case = Case(**cfg)
    d = case.d
    want = case.run(case.step(), d["l0"], d["l1"])
    got = case.run(case.step(), d["l0"], d["l1"], noise_seed=SEED, noise_level=0.0)
    _same(got[0], want[0], f"{name} forward")
    _same(got[1], want[1], f"{name} backward")


def test_batch_of_256_equals_two_batches_of_128(ups):
    """The draw follows the global sample index: a B=256 step equals two B=128 steps with sample_offset 0 and 128,
    per pixel bit for bit (the per-sample sums pooled and dfeat use the split geometry of their own batch size)."""
    B, S, K, F = 256, 128, 16, 64
    case = Case(B, S, K, F, seed=9)
    d = case.d
    whole = case.run(case.step(), d["l0"], d["l1"], noise_seed=SEED, noise_level=1.0)
    for h in range(2):
        lo, hi = 128 * h, 128 * (h + 1)
        sub = Case(128, S, K, F, seed=9)
        sub.d = dict(d, views=d["views"][:, lo:hi].contiguous(), l0=d["l0"][lo:hi], l1=d["l1"][lo:hi], feat=d["feat"][lo:hi],
                     coord=torch.cat([d["coord"][lo:hi], d["coord"][B + lo:B + hi]]),
                     t_vector=torch.cat([d["t_vector"][lo:hi], d["t_vector"][B + lo:B + hi]]),
                     cot=dict(d["cot"], g_inj=d["cot"]["g_inj"][lo:hi], g_pooled=d["cot"]["g_pooled"][lo:hi],
                              g_m0=d["cot"]["g_m0"][lo:hi], g_m1=d["cot"]["g_m1"][lo:hi]))
        sub.g1 = sub.d["cot"]["g_inj"]
        sub.g2 = d["cot"]["g_parts"].reshape(K, B, S, S, 3)[:, lo:hi].reshape(K * 128, S, S, 3).contiguous()
        out, grad = sub.run(sub.step(sample_offset=lo), sub.d["l0"], sub.d["l1"], noise_seed=SEED, noise_level=1.0)
        for k in ("m0", "m1", "labels0", "inj"):
            assert torch.equal(out[k], whole[0][k][lo:hi]), (h, k)
        assert torch.equal(out["parts"], whole[0]["parts"].reshape(K, B, S, S, 3)[:, lo:hi].reshape(K * 128, S, S, 3)), h
        for k in ("dl0", "dl1"):
            assert torch.equal(grad[k], whole[1][k][lo:hi]), (h, k)


def test_k25_parts_equal_k32_lanes(ups):
    """K=25 draws what K=32 draws for parts 0..24: the K=25 step on means equals the K=32 step on the same means padded
    with -inf (the padded parts stay -inf after the noise)."""
    B, S, F = 3, 64, 64
    e25, e32 = _eps(B, S, 25, 0), _eps(B, S, 32, 0)
    assert_bitexact(e25, e32[..., :25].contiguous(), "eps K=25 vs K=32")
    c25 = Case(B, S, 25, F, seed=4)
    out25, _ = c25.run(c25.step(), c25.d["l0"], c25.d["l1"], noise_seed=SEED, noise_level=LEVEL)
    c32 = Case(B, S, 32, F, seed=4)
    pad = lambda t: torch.cat([t, torch.full(t.shape[:-1] + (7,), float("-inf"), device="cuda")], -1).contiguous()  # noqa: E731
    feat = torch.cat([c25.d["feat"], torch.zeros(B, 7, F, device="cuda")], 1).contiguous()
    c32.d = dict(c25.d, l0=pad(c25.d["l0"]), l1=pad(c25.d["l1"]), feat=feat)
    c32.g1 = torch.zeros(B, S, S, F + 32, device="cuda")
    c32.g2 = torch.zeros(32 * B, S, S, 3, device="cuda")
    c32.d["cot"] = dict(c25.d["cot"], g_pooled=None, g_m0=None, g_m1=None)
    out32, _ = c32.run(c32.step(), c32.d["l0"], c32.d["l1"], noise_seed=SEED, noise_level=LEVEL)
    for k in ("m0", "m1"):
        assert_bitexact(out32[k][..., :25].contiguous(), out25[k], k)
        assert not out32[k][..., 25:].any()
    assert torch.equal(out32["labels0"], out25["labels0"])


def test_two_runs_give_identical_outputs(ups):
    case = Case(4, 128, 16, 64, seed=6)
    step = case.step()
    a = case.run(step, case.d["l0"], case.d["l1"], noise_seed=SEED)
    b = case.run(step, case.d["l0"], case.d["l1"], noise_seed=SEED)
    _same(b[0], a[0], "forward")
    _same(b[1], a[1], "backward")
    c = case.run(step, case.d["l0"], case.d["l1"], noise_seed=SEED + 1)
    assert not torch.equal(c[0]["m0"], a[0]["m0"])


def test_data_parallel_world1_passes_the_seed(ups):
    from ups_b200.dp import DataParallelPartStep
    case = Case(4, 64, 16, 64, seed=8)
    d = case.d
    dp = DataParallelPartStep(4, 64, 16, 64, n_views=3, n_grad_params=100_000, standin=True)
    assert dp.step.sample_offset == 0
    out = _clone(dp.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"], noise_seed=SEED,
                            noise_level=LEVEL))
    torch.cuda.synchronize()
    want, _ = case.run(case.step(), d["l0"], d["l1"], noise_seed=SEED, noise_level=LEVEL)
    _same(out, want, "dp forward")
