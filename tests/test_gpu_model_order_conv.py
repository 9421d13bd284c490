"""-m gpu: the step's two sides with their first convolutions folded in (SURVEY 8f N4), as differentiable ops in the
reference model's order: model.encode_conv2d (ups::encode_conv) and model.decode_conv2d with a noise seed
(ups::decode_conv).

  1. the ops produce the bits of PartStep(first_conv=Co, encoder_conv=Ce), forward and backward, with and without noise,
     at CUB B=256 K=16 and K=25 (e0 past 2^31 elements) and at a small K=8;
  2. a tiny model through the folded ops equals the same model through part_encode / part_decode and cuDNN convolutions;
  3. the noise seed: device == int, a new value redraws, noise_level=0 is noise-free, batches split at sample_offset;
  4. one captured CUDA graph of a training step, an int seed during capture, opcheck, torch.compile(fullgraph=True);
  5. errors (image gradient, K=40) and two micro-batches before their backwards.

The module prints its peak device memory (pytest -s)."""
import pytest
import torch

from util import assert_close, own_error_atol
from util import assert_bitexact as _assert_bitexact

pytestmark = pytest.mark.gpu

SEED, LEVEL = 0x5EED_0123_4567_89AB, 0.7


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    torch.cuda.reset_peak_memory_stats()
    yield ups_b200
    print(f"\ntest_gpu_model_order_conv: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


@pytest.fixture
def deterministic():
    prev = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
            torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
     torch.backends.cuda.matmul.allow_tf32) = prev


@pytest.fixture(autouse=True)
def _free_between_cases():
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def assert_bitexact(got, want, what=""):
    """util.assert_bitexact with the comparison on the device: the reference is copied to the host only on a mismatch."""
    if not torch.equal(got.detach().contiguous().view(torch.int32), want.detach().contiguous().view(torch.int32)):
        _assert_bitexact(got, want.detach().cpu(), what)


def _seed_tensor(seed):
    from ups_b200 import ops
    return torch.tensor([ops._seed_i64(seed)], dtype=torch.int64, device="cuda")


def _inputs(B, S, K, F, Co, Ce, seed):
    """Inputs and cotangents drawn on the device; exact ties (rounded logits) in row 0 of l0 and all-equal logits in row 1
    of l1, which give multi-hot masks (the dense paths of the convolutions)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)  # noqa: E731
    d = dict(img1=torch.rand(B, S, S, 3, device="cuda", generator=g) * 2 - 1, l0=r(B, S, S, K), l1=r(B, S, S, K),
             feat=r(B, K, F), Vd=r(3, 3, F + K, Co) * 0.05, bd=r(Co) * 0.1, Ve=r(3, 3, 3, Ce) * 0.2, be=r(Ce) * 0.1)
    d["l0"][:, 0] = torch.round(d["l0"][:, 0])
    d["l1"][:, 1] = 0.0
    d["cot"] = dict(g_h0=r(B, S, S, Co), g_e0=r(K * B, S, S, Ce), g_m0=r(B, S, S, K), g_m1=r(B, S, S, K))
    return d


# ---------------------------------------------------------------- 1. the bits of PartStep
# (name, B, S, K, F, Co, Ce)
CASES = [
    ("cub_b256_k16", 256, 128, 16, 64, 32, 32),       # bench.py's N4 leg
    ("cub_b256_k25", 256, 128, 25, 64, 32, 32),       # the shipped part count: e0 holds 25*256*128^2*32 > 2^31 floats
    ("k8", 2, 64, 8, 32, 16, 8),
]


def _ids():
    return [pytest.param(c, nz, id=f"{c[0]}-{nz}") for c in CASES for nz in ("none", "int", "device")
            if nz == "none" or c[3] in (16, 25)]


def _partstep(d, B, S, K, F, Co, Ce, seed):
    """PartStep's outputs and its two backwards (all cotangents; only g_h0 and g_e0).  The step and its buffers are
    freed before returning: what is returned is the step's e0 and clones of everything else."""
    from ups_b200.step import PartStep
    c = d["cot"]
    step = PartStep(B, S, K, F, n_views=2, use_tps=False, first_conv=Co, encoder_conv=Ce)
    views = torch.stack([d["img1"], d["img1"]])
    o = step.forward(views, None, None, d["l0"], d["l1"], d["feat"], d["Vd"], d["bd"], d["Ve"], d["be"],
                     noise_seed=seed, noise_level=LEVEL)
    want = {k: o[k].clone() for k in ("m0", "m1", "labels0", "h0")}
    want.update(e0=o["e0"], mask0=step.mh0c.clone(), mask1=step.mh1c.clone())
    g = step.backward(c["g_h0"], c["g_e0"], None, c["g_m0"], c["g_m1"])
    want.update({k: g[k].clone() for k in ("dl0", "dl1", "dfeat", "dV", "db", "dVe", "dbe")})
    g = step.backward(c["g_h0"], c["g_e0"])
    only = {k: g[k].clone() for k in ("dl0", "dl1", "dfeat", "dV", "db", "dVe", "dbe")}
    del step, o, g, views
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return want, only


@pytest.mark.parametrize("case,nz", _ids())
def test_ops_equal_partstep(ups, case, nz):
    name, B, S, K, F, Co, Ce = case
    d = _inputs(B, S, K, F, Co, Ce, seed=11)
    want, only = _partstep(d, B, S, K, F, Co, Ce, None if nz == "none" else SEED)
    leaves = {k: d[k].clone().requires_grad_() for k in ("l0", "l1", "feat", "Vd", "bd", "Ve", "be")}
    noise_seed = None if nz == "none" else SEED if nz == "int" else _seed_tensor(SEED)
    m1, mask1, e0 = ups.model.encode_conv2d(leaves["l1"], d["img1"], leaves["Ve"], leaves["be"], noise_seed, LEVEL)
    m0, labels0, mask0, h0 = ups.model.decode_conv2d(leaves["l0"], leaves["feat"], leaves["Vd"], leaves["bd"], noise_seed,
                                                     LEVEL)
    got = dict(m0=m0, m1=m1, labels0=labels0, h0=h0, e0=e0, mask0=mask0, mask1=mask1)
    for k in got:
        if k == "labels0":
            assert torch.equal(got[k], want[k]), (name, nz, k)
        else:
            assert_bitexact(got[k], want[k], f"{name}/{nz}: {k}")
    del want["e0"]
    c = d["cot"]
    xs = [leaves[k] for k in ("l0", "l1", "feat", "Vd", "bd", "Ve", "be")]
    names = ("dl0", "dl1", "dfeat", "dV", "db", "dVe", "dbe")
    gs = torch.autograd.grad([h0, e0, m0, m1], xs, [c["g_h0"], c["g_e0"], c["g_m0"], c["g_m1"]], retain_graph=True)
    for k, v in zip(names, gs):
        assert_bitexact(v, want[k], f"{name}/{nz}: {k}")
    # only h0 and e0 reach the loss: the cotangents of m0, m1 and the masks are undefined
    gs = torch.autograd.grad([h0, e0], xs, [c["g_h0"], c["g_e0"]])
    for k, v in zip(names, gs):
        assert_bitexact(v, only[k], f"{name}/{nz}, h0 and e0 only: {k}")


# ---------------------------------------------------------------- 2. the fold equals the unfolded model
class Tiny(torch.nn.Module):
    """e_pi: one 3x3 convolution from a warped view to part logits; e_alpha: its first layer (Ve, be) on the part images,
    relu, mean pool and a linear layer; dd: its first layer (Vd, bd) on the injected map, relu and a 3x3 convolution to
    RGB.  The first layers are TensorFlow-layout (HWIO) parameters, folded (encode_conv2d / decode_conv2d) or applied
    by cuDNN to the part images and the injected map of part_encode / part_decode."""

    def __init__(self, K, F, Ce, Co, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        self.K, self.F, self.Ce = K, F, Ce
        self.e_pi = torch.nn.Conv2d(3, K, 3, padding=1)
        self.Ve = torch.nn.Parameter(torch.randn(3, 3, 3, Ce) * 0.2)
        self.be = torch.nn.Parameter(torch.randn(Ce) * 0.1)
        self.lin = torch.nn.Linear(Ce, F)
        self.Vd = torch.nn.Parameter(torch.randn(3, 3, F + K, Co) * 0.05)
        self.bd = torch.nn.Parameter(torch.randn(Co) * 0.1)
        self.out = torch.nn.Conv2d(Co, 3, 3, padding=1)

    @staticmethod
    def nchw(x):
        return x.permute(0, 3, 1, 2)

    @staticmethod
    def nhwc(x):
        return x.permute(0, 2, 3, 1).contiguous()

    def conv_hwio(self, x, V, b):
        return self.nhwc(torch.nn.functional.conv2d(self.nchw(x), V.permute(3, 2, 0, 1), b, padding=1))

    def forward(self, views, fused, noise_seed=None, level=1.0, taps=None):
        from ups_b200 import model as M
        v0, v1, v0t = views
        B = v0.shape[0]
        l0 = self.nhwc(self.e_pi(self.nchw(v0)))
        l1 = self.nhwc(self.e_pi(self.nchw(v1)))
        if fused:
            m1, mask1, e0 = M.encode_conv2d(l1, v1, self.Ve, self.be, noise_seed, level)
        else:
            m1, parts, _ = M.part_encode(l1, v1, noise_seed, level)
            e0 = self.conv_hwio(parts, self.Ve, self.be)
        feat = self.lin(torch.relu(e0).mean(dim=(1, 2))).view(self.K, B, self.F).transpose(0, 1).contiguous()
        if fused:
            m0, labels0, mask0, h0 = M.decode_conv2d(l0, feat, self.Vd, self.bd, noise_seed, level)
        else:
            m0, labels0, inj = M.part_decode(l0, feat, noise_seed, level)
            h0 = self.conv_hwio(inj, self.Vd, self.bd)
        if taps is not None:
            for name, t in (("l0", l0), ("l1", l1), ("feat", feat)):
                t.register_hook(lambda g, name=name: taps.__setitem__("d" + name, g.clone()))
        rec = self.nhwc(self.out(self.nchw(torch.relu(h0))))
        loss = (rec - v0t).square().mean() + M.categorical_kl(m0) + M.categorical_kl(m1)
        return loss, dict(m0=m0, m1=m1, labels0=labels0, e0=e0, h0=h0, feat=feat)

    def forward64(self, views, m0_32, m1_32):
        """The unfolded model in float64 with plain torch ops; the hard masks (discrete decisions) are the fp32 ones."""
        v0, v1, v0t = (v.double() for v in views)
        B = v0.shape[0]
        p = {n: t.double() for n, t in self.named_parameters()}
        conv = lambda x, w, b: self.nhwc(torch.nn.functional.conv2d(self.nchw(x), w, b, padding=1))  # noqa: E731
        l0, l1 = conv(v0, p["e_pi.weight"], p["e_pi.bias"]), conv(v1, p["e_pi.weight"], p["e_pi.bias"])
        m0, m1 = torch.softmax(l0, -1), torch.softmax(l1, -1)
        hard = lambda m32: (m32 == m32.max(-1, keepdim=True).values).double()  # noqa: E731
        mask0, mask1 = hard(m0_32) + m0 - m0.detach(), hard(m1_32) + m1 - m1.detach()     # straight-through
        parts = (v1[:, :, :, None, :] * mask1[..., None]).permute(3, 0, 1, 2, 4).reshape(self.K * B, *v1.shape[1:])
        e0 = conv(parts, p["Ve"].permute(3, 2, 0, 1), p["be"])
        feat = (torch.relu(e0).mean(dim=(1, 2)) @ p["lin.weight"].T + p["lin.bias"]).view(self.K, B, self.F).transpose(0, 1)
        inj = torch.cat([torch.einsum("bhwk,bkf->bhwf", mask0, feat), mask0], -1)
        h0 = conv(inj, p["Vd"].permute(3, 2, 0, 1), p["bd"])
        rec = conv(torch.relu(h0), p["out.weight"], p["out.bias"])
        kl = lambda m: (m * torch.log(self.K * m + 1e-20)).sum(-1).mean()  # noqa: E731
        loss = (rec - v0t).square().mean() + kl(m0) + kl(m1)
        return loss, p


def _views(B, S, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(B, S, S, 3, generator=g) * 2 - 1).cuda() for _ in range(3)]


@pytest.mark.parametrize("K", [25, 16])
def test_fold_equals_unfolded_model(ups, deterministic, K):
    B, S, F, Ce, Co = 4, 64, 32, 16, 16
    views = _views(B, S, 4)
    res = []
    for fused in (True, False):
        model = Tiny(K, F, Ce, Co).cuda()
        loss, out = model(views, fused, SEED, LEVEL)
        loss.backward()
        res.append((loss.detach(), out, {n: p.grad.clone() for n, p in model.named_parameters()}))
    (lf, of, gf), (lu, ou, gu) = res
    for k in ("m0", "m1"):
        assert_bitexact(of[k], ou[k], k)
    assert torch.equal(of["labels0"], ou["labels0"])
    for k in ("e0", "feat", "h0"):
        assert_close(of[k], ou[k].cpu(), k)
    assert_close(lf, lu.cpu(), "loss")
    # the same model in float64 (noise-free: the fp32 runs' m0 / m1 under noise are softmaxes of the sampled logits, so
    # the float64 comparison uses a noise-free pair of fp32 runs)
    res = []
    for fused in (True, False):
        model = Tiny(K, F, Ce, Co).cuda()
        loss, out = model(views, fused)
        loss.backward()
        res.append((out, {n: p.grad.clone() for n, p in model.named_parameters()}))
    (of, gf), (ou, gu) = res
    model = Tiny(K, F, Ce, Co).cuda()
    loss64, p64 = model.forward64(views, ou["m0"], ou["m1"])
    g64 = dict(zip(p64, torch.autograd.grad(loss64, list(p64.values()))))
    for n in gu:       # every parameter gradient is a sum over the batch and the pixels
        atol = own_error_atol(gu[n], g64[n])
        assert_close(gf[n], g64[n].cpu(), f"grad {n} (float64)", atol=atol)
        assert_close(gf[n], gu[n].cpu(), f"grad {n} (fp32, unfolded)", atol=atol)


# ---------------------------------------------------------------- 3. seeds
def _both(ups, d, seed, level=LEVEL, offset=0, sl=slice(None)):
    m1, mask1, e0 = ups.model.encode_conv2d(d["l1"][sl], d["img1"][sl], d["Ve"], d["be"], seed, level, offset)
    m0, labels0, mask0, h0 = ups.model.decode_conv2d(d["l0"][sl], d["feat"][sl], d["Vd"], d["bd"], seed, level, offset)
    return dict(m0=m0, labels0=labels0, mask0=mask0, h0=h0, m1=m1, mask1=mask1, e0=e0)


def _equal(a, b, what):
    for k in a:
        assert torch.equal(a[k], b[k]), f"{what}: {k}"


@pytest.mark.parametrize("K", [16, 25])
def test_seeds(ups, K):
    from ups_b200 import ops
    B, S, F, Co, Ce = 4, 64, 32, 16, 8
    d = _inputs(B, S, K, F, Co, Ce, seed=3)
    seed_t = _seed_tensor(SEED)
    by_value = _both(ups, d, SEED)
    _equal(_both(ups, d, seed_t), by_value, "device seed vs int seed")
    clean = _both(ups, d, None)
    assert not torch.equal(by_value["m0"], clean["m0"]) and not torch.equal(by_value["m1"], clean["m1"])
    seed_t.fill_(ops._seed_i64(SEED + 1))
    redrawn = _both(ups, d, seed_t)
    for k in ("m0", "m1"):
        assert not torch.equal(redrawn[k], by_value[k]), f"a new value in the seed tensor must change the draw of {k}"
    _equal(_both(ups, d, SEED + 1), redrawn, "device seed vs int seed after the write")
    _equal(_both(ups, d, SEED, level=0.0), clean, "noise_level=0")
    _equal(_both(ups, d, seed_t, level=0.0), clean, "noise_level=0, device seed")
    # a batch of 2n = two batches of n at sample_offset 0 and n (a data-parallel split)
    n = B // 2
    whole = _both(ups, d, seed_t)
    halves = [_both(ups, d, seed_t, offset=o, sl=slice(o, o + n)) for o in (0, n)]
    for i, h in enumerate(halves):
        part = slice(i * n, (i + 1) * n)
        for k in h:
            w = whole[k].view(K, B, *whole[k].shape[1:])[:, part] if k == "e0" else whole[k][part]
            got = h[k].view(K, n, *h[k].shape[1:]) if k == "e0" else h[k]
            assert torch.equal(got, w), f"half {i}: {k}"
    assert not torch.equal(_both(ups, d, seed_t, offset=0, sl=slice(n, B))["m0"], halves[1]["m0"]), \
        "the second half must draw at its own sample_offset"


# ---------------------------------------------------------------- 4. graphs and compilation
def test_cuda_graph_step_equals_eager(ups, deterministic):
    from ups_b200 import ops
    B, S, K, F, Ce, Co = 2, 64, 25, 32, 16, 16
    views = _views(B, S, 6)
    model = Tiny(K, F, Ce, Co, seed=1).cuda()
    seed_t = _seed_tensor(0)
    static = {}
    params = ("Ve", "be", "Vd", "bd")

    def run(seed):
        taps = {}
        loss, out = model(views, True, seed, LEVEL, taps)
        loss.backward()
        return {**{k: out[k] for k in ("m0", "m1", "labels0", "e0", "h0")}, **taps}

    def grads():
        return {n: p.grad.clone() for n, p in model.named_parameters() if n in params}

    def eager(value):
        model.zero_grad(set_to_none=True)
        seed_t.fill_(ops._seed_i64(value))
        r = {k: v.clone() for k, v in run(seed_t).items()}
        r.update(grads())
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
    values = (3, SEED, 2 ** 64 - 5)
    results = []
    for value in values:
        seed_t.fill_(ops._seed_i64(value))
        graph.replay()
        torch.cuda.synchronize()
        results.append({**{k: v.clone() for k, v in static.items()}, **grads()})
    for value, got in zip(values, results):
        want = eager(value)
        for k in want:
            if want[k].dtype == torch.float32:
                assert_bitexact(got[k], want[k], f"seed={value}: {k}")
            else:
                assert torch.equal(got[k], want[k]), (value, k)
    assert not torch.equal(results[0]["m1"], results[1]["m1"]), "replays with different seeds must draw differently"


def test_int_seed_raises_during_capture(ups):
    from ups_b200 import _cabi as C
    B, S, K, F, Co, Ce = 2, 32, 16, 32, 16, 8
    d = _inputs(B, S, K, F, Co, Ce, seed=2)
    _both(ups, d, 1)                                      # warm-up outside capture
    for side in ("encode", "decode"):
        g = torch.cuda.CUDAGraph()
        with pytest.raises(C.UpsError, match="captured CUDA graph"):
            with torch.cuda.graph(g):
                if side == "encode":
                    ups.model.encode_conv2d(d["l1"], d["img1"], d["Ve"], d["be"], 1)
                else:
                    ups.model.decode_conv2d(d["l0"], d["feat"], d["Vd"], d["bd"], 1)


@pytest.mark.parametrize("K", [16, 25])
def test_opcheck(ups, K):
    from ups_b200 import ops
    B, S, F, Co, Ce = 2, 32, 32, 16, 8
    d = _inputs(B, S, K, F, Co, Ce, seed=8)
    l0, l1 = (d[k].clone().requires_grad_() for k in ("l0", "l1"))
    Ve, be, bd = (d[k].clone().requires_grad_() for k in ("Ve", "be", "bd"))
    G = ops.inject_conv_table(d["feat"], d["Vd"].reshape(9, F + K, Co)).detach().requires_grad_()
    Ve9 = Ve.detach().reshape(9, 3, Ce).requires_grad_()
    for args in ((l1, d["img1"], Ve9, be, ops.NOISE_NONE, None, 0, 1.0, 0),
                 (l1, d["img1"], Ve9, be, ops.NOISE_DEVICE, _seed_tensor(SEED), 0, LEVEL, 1),
                 (l1, d["img1"], Ve9, be, ops.NOISE_INT, None, 77, LEVEL, 0)):
        torch.library.opcheck(ops.encode_conv, args)
    for args in ((l0, G, bd), (l0, G, bd, ops.NOISE_INT, None, 77, LEVEL, 0),
                 (l0, G, bd, ops.NOISE_DEVICE, _seed_tensor(SEED), 0, LEVEL, 1)):
        torch.library.opcheck(ops.decode_conv, args)


def test_torch_compile_fullgraph(ups, deterministic):
    B, S, K, F, Co = 2, 64, 25, 16, 16
    d = _inputs(B, S, K, F, Co, F, seed=12)
    seed_t = _seed_tensor(SEED)

    def fn(l0, l1, img, seed, Ve, be, Vd, bd):
        m1, mask1, e0 = ups.model.encode_conv2d(l1, img, Ve, be, seed, LEVEL)
        feat = torch.relu(e0).mean(dim=(1, 2)).view(K, B, F).transpose(0, 1).contiguous()
        m0, labels0, mask0, h0 = ups.model.decode_conv2d(l0, feat, Vd, bd, seed, LEVEL)
        loss = h0.square().mean() + (m0 * m1).mean()
        return loss, m1, mask1, e0, m0, labels0, mask0, h0

    def step(f):
        xs = [d[k].clone().requires_grad_() for k in ("l0", "l1", "Ve", "be", "Vd", "bd")]
        out = f(xs[0], xs[1], d["img1"], seed_t, *xs[2:])
        out[0].backward()
        return out, [x.grad for x in xs]

    torch._dynamo.reset()
    got, got_g = step(torch.compile(fn, fullgraph=True))
    want, want_g = step(fn)
    for i in (1, 2, 3, 4, 5, 6):                  # m1, mask1, e0, m0, labels0, mask0: no compiled arithmetic before them
        assert torch.equal(got[i], want[i]), i
    assert_close(got[7], want[7].cpu(), "h0")
    assert_close(got[0], want[0].cpu(), "loss")
    for i, (a, b) in enumerate(zip(got_g, want_g)):
        assert_close(a, b.cpu(), f"grad {i}", atol=1e-5 + 1e-4 * float(b.abs().max()))


# ---------------------------------------------------------------- 5. errors and state
def test_image_gradient_raises(ups):
    from ups_b200 import _cabi as C
    d = _inputs(2, 32, 16, 32, 16, 8, seed=1)
    l1 = d["l1"].clone().requires_grad_()
    img = d["img1"].clone().requires_grad_()
    m1, mask1, e0 = ups.model.encode_conv2d(l1, img, d["Ve"], d["be"])
    with pytest.raises(C.UpsError, match="image"):
        e0.sum().backward()


def test_k40_raises(ups):
    from ups_b200 import _cabi as C
    d = _inputs(2, 32, 40, 32, 16, 8, seed=1)
    with pytest.raises(C.UpsError):
        ups.model.encode_conv2d(d["l1"], d["img1"], d["Ve"], d["be"])
    with pytest.raises(C.UpsError):
        ups.model.decode_conv2d(d["l0"], d["feat"], d["Vd"], d["bd"])


def test_two_forwards_then_two_backwards(ups, deterministic):
    B, S, K, F, Ce, Co = 2, 64, 25, 32, 16, 16
    model = Tiny(K, F, Ce, Co, seed=2).cuda()
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
