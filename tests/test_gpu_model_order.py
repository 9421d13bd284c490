"""-m gpu: the step's two sides as differentiable ops in the reference model's order (model.part_encode / part_decode,
ups::part_encode / ups::part_decode) and the noise seed read from device memory (the `_dseed` entry points).

  a. the ops produce the bits of PartStep (forward and backward) on every kernel route, with and without noise;
  b. a device seed draws exactly what the same value passed by value draws, for all four `_dseed` entry points;
  c. a tiny model trained through the ops has the gradients of the same model on the unfused reference-named ops;
  d. a whole training step captured in one CUDA graph redraws with the value in the seed tensor at every replay;
  e. torch.library.opcheck; f. torch.compile(fullgraph=True); g. two forwards before their backwards."""
import pytest
import torch

from util import assert_close, cuda, make_inputs
from util import assert_bitexact as _assert_bitexact

pytestmark = pytest.mark.gpu

SEED, LEVEL = 0x5EED_0123_4567_89AB, 0.7


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


def assert_bitexact(got, want, what=""):
    """util.assert_bitexact with the comparison on the device: the reference is copied to the host only on a mismatch,
    to report it."""
    if not torch.equal(got.detach().contiguous().view(torch.int32), want.detach().contiguous().view(torch.int32)):
        _assert_bitexact(got, want.detach().cpu(), what)


def _seed_tensor(seed):
    from ups_b200 import ops
    return torch.tensor([ops._seed_i64(seed)], dtype=torch.int64, device="cuda")


# ---------------------------------------------------------------- a. the bits of PartStep
# (name, B, S, K, F, PartStep decode_bwd, route, K4 on the tensor cores)
CASES = [
    ("cub_b256_k16_tc", 256, 128, 16, 64, "auto", "fused", True),
    ("k16_simt", 4, 64, 16, 32, "auto", "fused", False),
    ("k32", 4, 64, 32, 64, "auto", "fused", True),
    ("k25_contiguous", 4, 64, 25, 64, "auto", "padded", True),
    ("k8", 4, 64, 8, 32, "auto", "fused", False),
    ("generic_k40", 2, 32, 40, 64, "auto", "generic", False),
]
NOISES = ["none", "int", "device"]


def _ids():
    out = []
    for c in CASES:
        for nz in NOISES:
            if nz == "none" or c[3] in (16, 25, 40):
                out.append(pytest.param(c, nz, id=f"{c[0]}-{nz}"))
    return out


def _ops_step(ups, d, nz, seed=SEED, level=LEVEL, want_dimg=True):
    """Forward + backward through model.part_encode / part_decode with PartStep's cotangents."""
    l0 = d["l0"].clone().requires_grad_()
    l1 = d["l1"].clone().requires_grad_()
    feat = d["feat"].clone().requires_grad_()
    img1 = d["views"][1].clone().requires_grad_(want_dimg)
    noise_seed = None if nz == "none" else seed if nz == "int" else _seed_tensor(seed)
    m1, parts, pooled = ups.model.part_encode(l1, img1, noise_seed, level)
    m0, labels0, inj = ups.model.part_decode(l0, feat, noise_seed, level)
    c = d["cot"]
    torch.autograd.backward([m0, inj, m1, parts, pooled], [c["g_m0"], c["g_inj"], c["g_m1"], c["g_parts"], c["g_pooled"]])
    out = dict(m0=m0, m1=m1, labels0=labels0, parts=parts, pooled=pooled, inj=inj, dl0=l0.grad, dl1=l1.grad,
               dfeat=feat.grad)
    if want_dimg:
        out["dimg1"] = img1.grad
    return out


@pytest.mark.parametrize("case,nz", _ids())
def test_ops_equal_partstep(ups, case, nz):
    from ups_b200.step import PartStep, decode_bwd_tc_ok, kernel_route
    name, B, S, K, F, dbwd, route, tc = case
    assert kernel_route(K, F, S * S)[0] == route and kernel_route(K, None, S * S)[0] == route
    Kr = kernel_route(K, F, S * S)[1]
    assert (route != "generic" and decode_bwd_tc_ok(Kr, F, S * S)) == tc
    d = cuda(make_inputs(B, S, K, F, V=2, seed=11, ties=True))
    step = PartStep(B, S, K, F, n_views=2, use_tps=False, views_grad=True, decode_bwd=dbwd)
    inner = step._inner if step.Kp else step
    assert inner.decode_bwd == ("tc" if tc else "simt")
    seed = None if nz == "none" else SEED
    o = step.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"], noise_seed=seed, noise_level=LEVEL)
    want = {k: o[k].clone() for k in ("m0", "m1", "labels0", "parts", "pooled", "inj")}
    c = d["cot"]
    g = step.backward(c["g_inj"], c["g_parts"], c["g_pooled"], c["g_m0"], c["g_m1"])
    want.update({k: g[k].clone() for k in ("dl0", "dl1", "dfeat")}, dimg1=inner.dimg1.clone())
    got = _ops_step(ups, d, nz)
    for k, v in want.items():
        if v.dtype == torch.float32:
            assert_bitexact(got[k], v, f"{name}/{nz}: {k}")
        else:
            assert torch.equal(got[k], v), (name, nz, k)


def test_undefined_cotangents_are_skipped(ups):
    """Only inj and parts reach the loss: g_m0, g_m1, g_pooled are undefined and the kernels get null pointers,
    which equals PartStep's backward without them (and equals zeros for them)."""
    from ups_b200.step import PartStep
    B, S, K, F = 2, 64, 25, 64
    d = cuda(make_inputs(B, S, K, F, V=2, seed=5))
    step = PartStep(B, S, K, F, n_views=2, use_tps=False)
    step.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"])
    want = {k: v.clone() for k, v in step.backward(d["cot"]["g_inj"], d["cot"]["g_parts"]).items()}
    l0, l1, feat = (d[k].clone().requires_grad_() for k in ("l0", "l1", "feat"))
    m1, parts, pooled = ups.model.part_encode(l1, d["views"][1])
    m0, labels0, inj = ups.model.part_decode(l0, feat)
    torch.autograd.backward([inj, parts], [d["cot"]["g_inj"], d["cot"]["g_parts"]])
    for k, t in (("dl0", l0), ("dl1", l1), ("dfeat", feat)):
        assert_bitexact(t.grad, want[k], k)


# ---------------------------------------------------------------- b. device seed == seed by value
@pytest.mark.parametrize("K", [16, 25])
def test_device_seed_equals_int_seed(ups, K):
    from ups_b200 import _cabi as C
    from ups_b200 import ops
    st = torch.cuda.current_stream().cuda_stream
    n, off = 4096 + 32, 777
    seed_t = _seed_tensor(SEED)
    mean = torch.randn(n, K, device="cuda")

    def normal(dev, value):
        out = torch.empty(n, K, device="cuda")
        if dev:
            C.call("ups_normal_philox_fwd_dseed", seed_t.data_ptr(), 1, off, n, K, out.data_ptr(), st)
        else:
            C.call("ups_normal_philox_fwd", value, 1, off, n, K, out.data_ptr(), st)
        return out

    def sampled(dev, value):
        lo, pr, hd = (torch.empty(n, K, device="cuda") for _ in range(3))
        lab = torch.empty(n, dtype=torch.int64, device="cuda")
        s = seed_t.data_ptr() if dev else value
        C.call("ups_part_softmax_sampled_philox_fwd_dseed" if dev else "ups_part_softmax_sampled_philox_fwd",
               mean.data_ptr(), s, 0, off, LEVEL, lo.data_ptr(), pr.data_ptr(), lab.data_ptr(), hd.data_ptr(), n, K, st)
        return lo, pr, lab, hd

    for value in (SEED, 12345):
        seed_t.fill_(ops._seed_i64(value))
        assert_bitexact(normal(True, value), normal(False, value), f"normal_philox seed={value}")
        for a, b in zip(sampled(True, value), sampled(False, value)):
            assert torch.equal(a, b), f"part_softmax_sampled_philox seed={value}"
    seed_t.fill_(ops._seed_i64(SEED))
    before = normal(True, None)
    seed_t.fill_(ops._seed_i64(SEED + 1))
    assert not torch.equal(before, normal(True, None)), "a new seed value must change the draw"

    # the step's kernels (ups_step_{decode,encode}_fwd_noise[_dseed]) through the ops, and the draw they make
    B, S, F = 2, 64, 64
    d = cuda(make_inputs(B, S, K, F, V=2, seed=9))
    seed_t.fill_(ops._seed_i64(SEED))
    dev = ups.model.part_decode(d["l0"], d["feat"], seed_t, LEVEL, 3) + ups.model.part_encode(d["l1"], d["views"][1], seed_t,
                                                                                              LEVEL, 3)
    val = ups.model.part_decode(d["l0"], d["feat"], SEED, LEVEL, 3) + ups.model.part_encode(d["l1"], d["views"][1], SEED,
                                                                                            LEVEL, 3)
    for a, b in zip(dev, val):
        assert torch.equal(a, b)
    # ups_normal_philox_fwd_dseed regenerates what the step drew: the noise-free op on mean + level * eps
    for draw, (fn, arg, mean_) in enumerate(((ups.model.part_decode, d["feat"], d["l0"]),
                                            (ups.model.part_encode, d["views"][1], d["l1"]))):
        eps = torch.empty(B * S * S, K, device="cuda")
        C.call("ups_normal_philox_fwd_dseed", seed_t.data_ptr(), draw, 3 * S * S, B * S * S, K, eps.data_ptr(), st)
        logits = ops.mean_field_sample(mean_, eps.view(B, S, S, K), LEVEL)
        for a, b in zip(fn(logits, arg), dev[3 * draw:3 * draw + 3]):
            assert torch.equal(a, b), f"draw {draw}"
    seed_t.fill_(ops._seed_i64(SEED + 1))
    assert not torch.equal(ups.model.part_decode(d["l0"], d["feat"], seed_t, LEVEL, 3)[0], dev[0])


def test_int_seed_raises_during_capture(ups):
    from ups_b200 import _cabi as C
    B, S, K, F = 2, 32, 16, 64
    d = cuda(make_inputs(B, S, K, F, V=2, seed=2))
    ups.model.part_decode(d["l0"], d["feat"], 1)          # warm-up outside capture
    g = torch.cuda.CUDAGraph()
    with pytest.raises(C.UpsError, match="captured CUDA graph"):
        with torch.cuda.graph(g):
            ups.model.part_decode(d["l0"], d["feat"], 1)


# ---------------------------------------------------------------- c. a tiny model: fused ops vs the unfused ops
class Tiny(torch.nn.Module):
    """e_pi / dv: one 3x3 convolution from a warped view to part logits; e_alpha: a 3x3 convolution on the part images,
    mean pool and a linear layer; dd: one 3x3 convolution on the injected map.  The pooled part colours enter the loss
    directly: they are sums over pixels whose rounding differs between K2 and the unfused pooling kernel, so feeding
    them into `feat` would keep inj from being compared bit for bit."""

    def __init__(self, K, F, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        self.K, self.F = K, F
        self.e_pi = torch.nn.Conv2d(3, K, 3, padding=1)
        self.e_alpha = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.lin = torch.nn.Linear(8, F)
        self.dd = torch.nn.Conv2d(F + K, 3, 3, padding=1)

    @staticmethod
    def nchw(x):
        return x.permute(0, 3, 1, 2)

    @staticmethod
    def nhwc(x):
        return x.permute(0, 2, 3, 1).contiguous()

    def forward(self, views, fused, noise_seed=None, level=1.0, taps=None):
        from ups_b200 import model as M
        from ups_b200 import nn as N
        from ups_b200 import pooling
        v0, v1, v0t = views
        B = v0.shape[0]
        l0 = self.nhwc(self.e_pi(self.nchw(v0)))
        l1 = self.nhwc(self.e_pi(self.nchw(v1)))
        if fused:
            m1, parts, pooled = M.part_encode(l1, v1, noise_seed, level)
        else:
            m1 = N.softmax(l1)
            mh1 = N.hard_max_straight_through(m1, 3)
            parts = M.mask_parts_partmajor(v1, mh1)
            pooled = pooling.part_mean_pool(v1, mh1)
        e = torch.relu(self.e_alpha(self.nchw(parts))).mean(dim=(2, 3))            # [K*B, 8]
        feat = self.lin(e).view(self.K, B, self.F).transpose(0, 1)
        feat = feat.contiguous()
        if fused:
            m0, labels0, inj = M.part_decode(l0, feat, noise_seed, level)
        else:
            m0 = N.softmax(l0)
            labels0 = N.argmax(m0, 3)
            inj = M.inject_features(feat, N.hard_max_straight_through(m0, 3))
        if taps is not None:
            for name, t in (("l0", l0), ("l1", l1), ("feat", feat)):
                t.register_hook(lambda g, name=name: taps.__setitem__("d" + name, g.clone()))
        rec = self.nhwc(self.dd(self.nchw(inj)))
        loss = (rec - v0t).square().mean() + M.categorical_kl(m0) + M.categorical_kl(m1) + 0.1 * pooled.square().mean()
        return loss, dict(m0=m0, m1=m1, labels0=labels0, parts=parts, pooled=pooled, inj=inj)


def _views(B, S, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(B, S, S, 3, generator=g) * 2 - 1).cuda() for _ in range(3)]


@pytest.fixture
def deterministic():
    prev = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev


@pytest.mark.parametrize("K", [25, 16], ids=["cub_shipped_k25", "k16"])
def test_autograd_fused_equals_unfused(ups, deterministic, K):
    from ups_b200 import configs
    cfg = configs.CUB_SHIPPED
    B, S, F = cfg.batch_size, cfg.spatial_size, cfg.local_app_size
    assert K != 25 or K == cfg.n_parts
    views = _views(B, S, 4)
    res = []
    for fused in (True, False):
        model = Tiny(K, F).cuda()
        loss, out = model(views, fused)
        loss.backward()
        res.append((loss.detach(), out, {n: p.grad.clone() for n, p in model.named_parameters()}))
    (lf, of, gf), (lu, ou, gu) = res
    for k in ("m0", "m1", "parts", "inj"):
        assert_bitexact(of[k], ou[k], k)
    assert torch.equal(of["labels0"], ou["labels0"])
    assert_close(of["pooled"], ou["pooled"].cpu(), "pooled")
    assert_close(lf, lu.cpu(), "loss")
    for n in gu:
        assert_close(gf[n], gu[n].cpu(), f"grad {n}")


# ---------------------------------------------------------------- d. one captured CUDA graph of a training step
@pytest.mark.parametrize("K", [25, 16])
def test_cuda_graph_redraws_per_replay(ups, deterministic, K):
    from ups_b200 import ops
    B, S, F = 2, 64, 32
    views = _views(B, S, 6)
    model = Tiny(K, F, seed=1).cuda()
    seed_t = _seed_tensor(0)
    static = {}

    def run(seed):
        taps = {}
        loss, out = model(views, True, seed, LEVEL, taps)
        loss.backward()
        return {**{k: out[k] for k in ("m0", "m1", "labels0")}, **taps}

    def eager(value):
        model.zero_grad(set_to_none=True)
        seed_t.fill_(ops._seed_i64(value))
        r = {k: v.clone() for k, v in run(seed_t).items()}
        torch.cuda.synchronize()
        return r

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            model.zero_grad(set_to_none=True)
            run(seed_t)
    torch.cuda.current_stream().wait_stream(side)
    model.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static.update(run(seed_t))
    results = []
    for value in (3, SEED, 2 ** 64 - 5):
        seed_t.fill_(ops._seed_i64(value))
        graph.replay()
        torch.cuda.synchronize()
        results.append({k: v.clone() for k, v in static.items()})
    for value, got in zip((3, SEED, 2 ** 64 - 5), results):
        want = eager(value)
        for k in ("m0", "m1", "labels0", "dl0", "dl1", "dfeat"):
            if want[k].dtype == torch.float32:
                assert_bitexact(got[k], want[k], f"seed={value}: {k}")
            else:
                assert torch.equal(got[k], want[k]), (value, k)
    assert not torch.equal(results[0]["m0"], results[1]["m0"]), "replays with different seeds must draw differently"


# ---------------------------------------------------------------- e. opcheck, f. torch.compile
@pytest.mark.parametrize("K", [16, 25])
def test_opcheck(ups, K):
    from ups_b200 import ops
    B, S, F = 2, 32, 32
    d = cuda(make_inputs(B, S, K, F, V=2, seed=8))
    l0, l1, feat = (d[k].clone().requires_grad_() for k in ("l0", "l1", "feat"))
    img = d["views"][1].clone().requires_grad_()
    for args in ((l1, img, ops.NOISE_NONE, None, 0, 1.0, 0), (l1, img, ops.NOISE_DEVICE, _seed_tensor(SEED), 0, LEVEL, 1)):
        torch.library.opcheck(ops.part_encode, args)
    for args in ((l0, feat, ops.NOISE_NONE, None, 0, 1.0, 0), (l0, feat, ops.NOISE_INT, None, 77, LEVEL, 0)):
        torch.library.opcheck(ops.part_decode, args)


def test_torch_compile_fullgraph(ups, deterministic):
    B, S, K, F = 2, 64, 25, 32
    d = cuda(make_inputs(B, S, K, F, V=2, seed=12))
    conv = torch.nn.Conv2d(3, F, 3, padding=1).cuda()
    seed_t = _seed_tensor(SEED)

    def fn(l0, l1, img, seed):
        m1, parts, pooled = ups.model.part_encode(l1, img, seed, LEVEL)
        e = conv(parts.permute(0, 3, 1, 2)).mean(dim=(2, 3)).view(K, B, F).transpose(0, 1).contiguous()
        return (m1, pooled) + ups.model.part_decode(l0, e, seed, LEVEL)

    torch._dynamo.reset()
    compiled = torch.compile(fn, fullgraph=True)
    got = compiled(d["l0"], d["l1"], d["views"][1], seed_t)
    want = fn(d["l0"], d["l1"], d["views"][1], seed_t)
    for i in (0, 2, 3):                               # m1, m0, labels0: the path outputs the convolution does not touch
        assert torch.equal(got[i], want[i]), i
    assert_close(got[1], want[1].cpu(), "pooled")
    assert_close(got[4], want[4].cpu(), "inj")


# ---------------------------------------------------------------- g. two micro-batches before their backwards
def test_two_forwards_then_two_backwards(ups, deterministic):
    B, S, K, F = 2, 64, 25, 32
    model = Tiny(K, F, seed=2).cuda()
    mb = [_views(B, S, 20), _views(B, S, 21)]
    seeds = [_seed_tensor(5), _seed_tensor(6)]

    def grads():
        return {n: p.grad.clone() for n, p in model.named_parameters()}

    model.zero_grad(set_to_none=True)
    model(mb[0], True, seeds[0], LEVEL)[0].backward()
    g0 = grads()
    model.zero_grad(set_to_none=True)
    model(mb[1], True, seeds[1], LEVEL)[0].backward()
    g1 = grads()
    model.zero_grad(set_to_none=True)
    losses = [model(mb[i], True, seeds[i], LEVEL)[0] for i in range(2)]
    losses[0].backward()
    h0 = grads()
    model.zero_grad(set_to_none=True)
    losses[1].backward()
    h1 = grads()
    for n in g0:
        assert_bitexact(h0[n], g0[n], f"micro-batch 0: {n}")
        assert_bitexact(h1[n], g1[n], f"micro-batch 1: {n}")
