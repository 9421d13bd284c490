"""-m gpu: the mask-statistics, prior and sampling kernels (SURVEY.md 8f N1-N3) and the spatial softmax at the batch sizes
bench.py runs, against float64 references.

The launch geometry of these kernels depends on B, P and K, and the small shapes of test_gpu_stats.py /
test_gpu_priors.py reach little of it: at the bench's sizes the grid-stride loops of the logit priors and of the weak
cross entropy wrap (about 55 iterations per thread at CUB B=256), their finalize kernels reduce more than 1024 partials,
the last pixel split of the mask moments and of Mumford-Shah is partial in every sample (CUB: 10 splits of 1639 pixels,
the last one 1633), and K = 25 (the reference's shipped n_parts) runs the scalar and generic kernels over whole batches.
The cases are the bench's workloads (bench.WORKLOADS: cub, deepfashion, pennaction), CUB with K = 25, and CUB K = 16
passed as a contiguous view 4 bytes past a 16-byte boundary, which sends K = 16 to the scalar kernels.  Every sample's
first and last 256 pixels hold tied, x40 and all-equal logit rows.

* Elementwise maps, bit for bit: Mumford-Shah r / smooth / contour, edge_set, mean_field_sample, part_softmax_sampled
  (logits, probabilities, labels, hard mask) and mask2rgb hot.  The oracle is evaluated on the device, one chunk of
  samples at a time: each of its steps is one eager PyTorch op, i.e. one kernel doing one correctly rounded IEEE binary32
  operation per element (no FMA contraction across ops, no flush of subnormals), which is exactly what the CPU does.
  _oracle checks that claim on the first two samples of every chunk against the CPU evaluation.
* Values and gradients against float64 at 1e-4 rel / 1e-5 abs, with the fp32 decisions (Mumford-Shah branches, hard
  labels) taken from the fp32 oracle.
* Long sums against float64 within util.own_error_atol of the plain fp32 torch evaluation of the same expression
  (TF32 off); categorical KL adds the documented error of __logf / __fdividef.
* Exact probes of the split geometry read the kernels' split counts from the public workspace query: Mumford-Shah sums
  of inputs on a 1/8 grid are exact in any order, and single-pixel deltas at every split edge give mu bit for bit.
"""
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from oracle import parts as OP
from oracle import priors as OR
from oracle import stats as OS
from util import ATOL, RTOL, own_error_atol

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    spec = importlib.util.spec_from_file_location("bench_priors_workloads_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


BENCH = _load_bench()


def _case(workload, K=None, misaligned=False):
    wl = BENCH.WORKLOADS[workload]
    return dict(B=wl["B"], S=wl["S"], K=K or wl["K"], misaligned=misaligned)


CASES = {name: _case(name) for name in sorted(BENCH.WORKLOADS)}
CASES.update({"cub-k25": _case("cub", K=25), "cub-misaligned": _case("cub", misaligned=True)})
# categorical_kl and mean_field_sample have vector kernels only and reject a misaligned pointer
ALIGNED_CASES = [n for n in CASES if not CASES[n]["misaligned"]]
TAIL = 256
CHUNK = 1 << 23    # elements per chunk of the float64 references


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


@pytest.fixture(autouse=True)
def _fp32_plain():
    """The fp32 evaluations that set own_error_atol's bound must be plain fp32, not TF32."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.fixture(autouse=True)
def _free_between_cases():
    yield
    import gc
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ inputs
def _adversarial(logits):
    """The first and the last 256 pixels of every sample: rounded logits (exact ties), logits x40 (near one-hot
    softmax) and all-equal rows, as test_gpu_workloads.py does."""
    B, S, _, K = logits.shape
    P = S * S
    f = logits.view(B, P, K)
    for base in (0, P - TAIL):
        f[:, base:base + 96] = torch.round(f[:, base:base + 96])
        f[:, base + 96:base + 192] *= 40
        f[:, base + 192:base + TAIL] = 0.0


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _logits(c, seed):
    x = torch.randn(c["B"], c["S"], c["S"], c["K"], device="cuda", generator=_gen(seed))
    _adversarial(x)
    return x


def _place(t, misaligned):
    """t, or for the misaligned case a contiguous copy whose data pointer is 4 bytes past a 16-byte boundary: the ops
    only call .contiguous(), so the kernels see that pointer and take their scalar paths."""
    if not misaligned:
        return t
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device=t.device)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4, v.data_ptr()
    return v


def _chunks(c):
    B, P, K = c["B"], c["S"] * c["S"], c["K"]
    cb = max(1, CHUNK // (P * K))
    return [slice(b0, min(B, b0 + cb)) for b0 in range(0, B, cb)]


def _splits(op, c, n_sums):
    """The kernel's split count per sample, from ups_workspace_bytes = B*splits*K*n_sums*4 + 256."""
    from ups_b200 import _cabi as C
    B, P, K = c["B"], c["S"] * c["S"], c["K"]
    n = (C.workspace_bytes(op, B, P, K, 0) - 256) / (B * K * n_sums * 4)
    assert n == int(n) and n >= 1, n
    n = int(n)
    per = -(-P // n)
    # the point of these cases: every sample's last split is partial
    assert P % per != 0, f"B={B} P={P}: {n} splits of {per} pixels divide P evenly"
    return n, per


# ------------------------------------------------------------------------------------------------ comparisons
def _bits(x):
    return x.contiguous().view(torch.int32) if x.dtype == torch.float32 else x


def _same_bits(got, want, what):
    if not torch.equal(_bits(got), _bits(want)):
        n = int((_bits(got) != _bits(want)).sum())
        raise AssertionError(f"{what}: {n}/{got.numel()} elements differ bitwise")


def _oracle(fn, *batched):
    """fn(*batched) evaluated on the device; on the first two samples it must give what the CPU gives, bit for bit."""
    out = fn(*batched)
    cpu = fn(*[t[:2].cpu() for t in batched])
    for o, w in zip(out if isinstance(out, tuple) else (out,), cpu if isinstance(cpu, tuple) else (cpu,)):
        _same_bits(o[:2].cpu(), w, f"device oracle != CPU oracle ({getattr(fn, '__name__', fn)})")
    return out


class _Bound:
    """Kernel output against its float64 value, accumulated chunk by chunk: passes when
    |kernel - f64| <= atol + RTOL |f64| + slack everywhere (atol may be a tensor), and for a long sum (check(own=True))
    within a further 2 max |fp32 - f64|, util.own_error_atol's measured bound."""

    def __init__(self, what):
        self.what, self.excess, self.own, self.at = what, -math.inf, 0.0, None

    def add(self, got, ref64, ref32=None, where=None, atol=ATOL, slack=0.0):
        e = float(((got.detach().double() - ref64).abs() - RTOL * ref64.abs() - atol - slack).max())
        if e > self.excess:
            self.excess, self.at = e, where
        if ref32 is not None:
            self.own = max(self.own, float((ref32.detach().double() - ref64).abs().max()))

    def check(self, own=False):
        allow = 2.0 * self.own if own else 0.0
        assert self.excess <= allow, (f"{self.what}: |kernel - float64| exceeds its tolerance by "
                                      f"{self.excess - allow:.3e} (samples {self.at})")


def _where(s):
    return f"{s.start}..{s.stop - 1}"


# ------------------------------------------------------------------------------------------------ Mumford-Shah
def _ms64(p, alpha, lam, le, lt, ge):
    """oracle.priors.mumford_shah in float64 with the branch decisions of the fp32 evaluation (ag <= lam, ag < lam,
    ag >= lam): the value and the tf.minimum / tf.where gradient routing the kernels implement."""
    right = torch.cat([p[:, :, 1:], torch.zeros_like(p[:, :, :1])], dim=2)
    down = torch.cat([p[:, 1:], torch.zeros_like(p[:, :1])], dim=1)
    gx, gy = 0.25 * (p - right), 0.25 * (p - down)
    ag = alpha * (gx * gx + gy * gy)
    r = torch.where(le, ag, lam)
    return r, torch.where(lt, r, 0.0), torch.where(ge, r, 0.0)


@pytest.mark.parametrize("name", list(CASES))
def test_mumford_shah(ups, name):
    c = CASES[name]
    B, K = c["B"], c["K"]
    p = _place(torch.softmax(_logits(c, 1), -1), c["misaligned"])
    alpha = 1.5
    lam = float(alpha * OR.tf_squared_grad(p[:8]).median())         # both branches of the minimum occur
    lam32 = torch.tensor(lam, dtype=torch.float32, device="cuda")
    pg = p.requires_grad_(True)
    maps = ups.nn.mumford_shah(pg, alpha, lam)
    edges = ups.nn.edge_set(p, alpha, lam)
    g = _gen(2)
    cots = [torch.randn(p.shape, device="cuda", generator=g) for _ in range(3)]
    (d,) = torch.autograd.grad(maps, pg, cots)
    sums = ups.nn.mumford_shah_sums(pg, alpha, lam)
    assert tuple(sums.shape) == (B, 4, K)
    g_sums = torch.randn(B, 4, K, device="cuda", generator=g)
    (ds,) = torch.autograd.grad(sums, pg, g_sums)
    torch.cuda.synchronize()
    names = ("r", "smoothness_cost", "contour_cost", "x")
    b_d, b_ds = _Bound("d x (elementwise cotangents)"), _Bound("d x (sum cotangents)")
    b_sum = [_Bound(f"sum of {n}") for n in names]
    for s in _chunks(c):
        pc = p[s].detach()
        want = _oracle(lambda t: OR.mumford_shah(t, alpha, lam), pc)
        for got, w, n in zip(maps, want, names):
            _same_bits(got[s], w, f"{n} (samples {_where(s)})")
        _same_bits(edges[s], _oracle(lambda t: OR.edge_set(t, alpha, lam), pc), f"edge_set (samples {_where(s)})")
        ag32 = alpha * OR.tf_squared_grad(pc)
        le, lt, ge = ag32 <= lam32, ag32 < lam32, ag32 >= lam32
        del ag32
        p64 = pc.double().requires_grad_(True)
        m64 = _ms64(p64, alpha, lam, le, lt, ge)
        (d64,) = torch.autograd.grad(m64, p64, [t[s].double() for t in cots])
        b_d.add(d[s], d64, where=_where(s))
        # the kernel sums the fp32 map values: their float64 sum is the exact value of that sum
        for i, v in enumerate((*want, pc)):
            b_sum[i].add(sums[s, i], v.double().sum((1, 2)), v.sum((1, 2)), where=_where(s))
        gs = g_sums[s].double()[:, :, None, None, :]
        m64 = _ms64(p64, alpha, lam, le, lt, ge)
        tot = sum((v * gs[:, i]).sum() for i, v in enumerate((*m64, p64)))
        (d64,) = torch.autograd.grad(tot, p64)
        b_ds.add(ds[s], d64, where=_where(s))
        del p64, m64, d64, tot, want
    b_d.check()
    b_ds.check()
    for b in b_sum:
        b.check(own=True)


@pytest.mark.parametrize("name", list(CASES))
def test_mumford_shah_sums_exact_at_split_edges(ups, name):
    """Inputs on the 1/8 grid of [0, 1], alpha = 1, lambda = 1/16: every term (a multiple of 2^-10 below 1/8, or of 1/8
    for x) and every partial sum (below 2^12, or 2^16 for x: at most 22 significant bits) is exact in fp32, so all four
    sums equal the float64 value bit for bit whatever the summation order.  A pixel dropped or added at a split edge
    changes them."""
    from ups_b200 import _cabi as C
    c = CASES[name]
    _splits(C.OP_MUMFORD_SHAH, c, 4)
    B, S, K = c["B"], c["S"], c["K"]
    q = torch.randint(0, 9, (B, S, S, K), device="cuda", generator=_gen(3)).float() / 8
    sums = ups.nn.mumford_shah_sums(_place(q, c["misaligned"]), 1.0, 1.0 / 16)
    torch.cuda.synchronize()
    for s in _chunks(c):
        want = OR.mumford_shah_sums(q[s].double(), 1.0, 1.0 / 16)
        assert torch.equal(sums[s].double(), want), (
            f"sums on the 1/8 grid != exact value (samples {_where(s)}): max |d| "
            f"{float((sums[s].double() - want).abs().max()):.3e}")


# ------------------------------------------------------------------------------------------------ mask moments
@pytest.mark.parametrize("name", list(CASES))
def test_mask_moments(ups, name):
    c = CASES[name]
    B, S, K = c["B"], c["S"], c["K"]
    dens = torch.softmax(_logits(c, 4).view(B, S * S, K), dim=1).view(B, S, S, K)    # sums to 1 over HW
    g = _gen(5)
    sf = torch.rand(B, K, device="cuda", generator=g) * 0.5 + 0.75
    dg = _place(dens, c["misaligned"]).requires_grad_(True)
    mu, sigma = ups.nn.probs_to_mu_sigma(dg, sf)
    assert tuple(mu.shape) == (B, K, 2) and tuple(sigma.shape) == (B, K, 2, 2)
    g_mu, g_sigma = torch.randn(B, K, 2, device="cuda", generator=g), torch.randn(B, K, 2, 2, device="cuda", generator=g)
    (dd,) = torch.autograd.grad([mu, sigma], dg, [g_mu, g_sigma])
    torch.cuda.synchronize()
    b_mu, b_sigma, b_dd = _Bound("mu"), _Bound("sigma"), _Bound("d probs")
    for s in _chunks(c):
        mu32, sigma32 = OS.probs_to_mu_sigma(dens[s], sf[s])
        d64 = dens[s].double().requires_grad_(True)
        mu64, sigma64 = OS.probs_to_mu_sigma(d64, sf[s].double())
        b_mu.add(mu[s], mu64.detach(), mu32, where=_where(s))
        b_sigma.add(sigma[s], sigma64.detach(), sigma32, where=_where(s))
        (dd64,) = torch.autograd.grad([mu64, sigma64], d64, [g_mu[s].double(), g_sigma[s].double()])
        b_dd.add(dd[s], dd64, where=_where(s))
        del d64, dd64
    b_mu.check(own=True)
    b_sigma.check(own=True)
    b_dd.check()


def _lin_at(i, n):
    """csrc/canon_math.cuh lin_step / lin_at in numpy float32: fl(-1 + fl(i * fl(2 / (n - 1))))."""
    step = np.float32(2.0) / np.float32(n - 1)
    return np.float32(-1.0) + np.asarray(i).astype(np.float32) * step


@pytest.mark.parametrize("name", list(CASES))
def test_mask_moments_deltas_at_split_edges(ups, name):
    """Every (b, k) plane is a single-pixel delta, placed in turn on the first and the last pixel of every split, the
    pixel before each split, and pixels 0 and P-1.  Then every partial sum is exact: mu must be fl(lin_at(i) * s) and
    fl(lin_at(j) * s) bit for bit, and sigma zero up to what an FMA-contracted m2 - m0^2 leaves, s^2 2^-23 |y y'|."""
    from ups_b200 import _cabi as C
    c = CASES[name]
    B, S, K = c["B"], c["S"], c["K"]
    P = S * S
    splits, per = _splits(C.OP_MOMENTS, c, 5)
    pos = sorted({0, P - 1} | {k * per for k in range(splits)} | {min((k + 1) * per, P) - 1 for k in range(splits)}
                 | {k * per - 1 for k in range(1, splits)})
    pix = np.asarray(pos)[np.arange(B * K) % len(pos)]
    dens = torch.zeros(B, P, K, device="cuda")
    dens[torch.arange(B).repeat_interleave(K), torch.from_numpy(pix).cuda(), torch.arange(K).repeat(B)] = 1.0
    sf = torch.rand(B, K, device="cuda", generator=_gen(6)) * 0.5 + 0.75
    mu, sigma = ups.nn.probs_to_mu_sigma(_place(dens.view(B, S, S, K), c["misaligned"]), sf)
    mu = mu.cpu().numpy().reshape(B * K, 2)
    sigma = sigma.cpu().numpy().reshape(B * K, 2, 2).astype(np.float64)
    s = sf.cpu().numpy().reshape(B * K)
    y, x = _lin_at(pix // S, S), _lin_at(pix % S, S)
    for axis, lin in ((0, y), (1, x)):
        want = lin * s
        bad = np.nonzero(mu[:, axis].view(np.int32) != want.view(np.int32))[0]
        assert bad.size == 0, (f"mu[..., {axis}] of {bad.size} deltas != fl(lin_at * s); first at pixel {pix[bad[0]]} "
                               f"(split {pix[bad[0]] // per} of {splits}, {per} pixels each): {mu[bad[0], axis]!r} "
                               f"vs {want[bad[0]]!r}")
    y64, x64, s64 = y.astype(np.float64), x.astype(np.float64), s.astype(np.float64)
    yy = np.stack([np.stack([y64 * y64, np.abs(y64 * x64)], -1), np.stack([np.abs(y64 * x64), x64 * x64], -1)], -2)
    bound = (s64 * s64)[:, None, None] * 2.0 ** -23 * yy
    bad = np.nonzero((np.abs(sigma) > bound).any((1, 2)))[0]
    assert bad.size == 0, f"sigma of {bad.size} deltas not zero; first at pixel {pix[bad[0]]}: {sigma[bad[0]]}"


# ------------------------------------------------------------------------------------------------ categorical KL
# __logf: absolute error at most 2^-21.41 for u in [0.5, 2], at most 3 ulp elsewhere; __fdividef: at most 2 ulp
# (CUDA C++ Programming Guide, intrinsic functions).  1 ulp of v is at most 2^-23 |v|.
def _logf_error(lg):
    return torch.clamp(3.0 * 2.0 ** -23 * lg.abs(), min=2.0 ** -21.41)


@pytest.mark.parametrize("name", ALIGNED_CASES)
def test_categorical_kl(ups, name):
    c = CASES[name]
    K = c["K"]
    p = torch.softmax(_logits(c, 7), -1)
    n_pix = p.numel() // K
    pg = p.requires_grad_(True)
    kl = ups.model.categorical_kl(pg)
    cot = 0.7 * n_pix                                                # keeps the gradient entries O(1)
    (dp,) = torch.autograd.grad(kl, pg, torch.tensor(cot, device="cuda"))
    kl32 = OS.categorical_kl(p.detach())
    torch.cuda.synchronize()
    g = cot / n_pix
    total64, slack = 0.0, 0.0
    b_dp = _Bound("d kl")
    for s in _chunks(c):
        p64 = p[s].detach().double()
        u = K * p64 + 1e-20
        lg = torch.log(u)
        total64 += float((p64 * lg).sum())
        # sum_k p_k = 1 per pixel: the mean over pixels of sum_k p_k err(log u_k) is at most the largest error of the log
        elog = _logf_error(lg)
        slack += float((p64 * elog).sum())
        q = K * p64 / u
        b_dp.add(dp[s], g * (lg + q), where=_where(s), slack=g * (elog + 2.0 * 2.0 ** -23 * q))
        del p64, u, lg, elog, q
    kl64 = total64 / n_pix
    atol = own_error_atol(kl32, torch.tensor(kl64)) + slack / n_pix
    err = abs(float(kl.detach()) - kl64)
    assert err <= atol + RTOL * abs(kl64), f"kl {float(kl.detach())!r} vs float64 {kl64!r}: |d| {err:.3e} > {atol:.3e} + rtol"
    b_dp.check()


# ------------------------------------------------------------------------------------------------ logit priors
@pytest.mark.parametrize("name", list(CASES))
def test_logit_priors(ups, name):
    """kl, kl_improper_gmrf, kl_tv: sums over B*H*W*K terms (grid-stride loops that wrap, more than 1024 partials)."""
    c = CASES[name]
    B = c["B"]
    x = _place(_logits(c, 8), c["misaligned"]).requires_grad_(True)
    pri = ups.ops.logit_priors(x)
    cot = torch.randn(3, device="cuda", generator=_gen(9)) * B      # keeps the gradient entries O(1)
    (d,) = torch.autograd.grad(pri, x, cot)
    pri32 = OR.logit_priors(x.detach())
    torch.cuda.synchronize()
    pri64 = torch.zeros(3, dtype=torch.float64, device="cuda")
    b_d = _Bound("d logits")
    for s in _chunks(c):
        x64 = x[s].detach().double().requires_grad_(True)
        w = (s.stop - s.start) / B                                   # the oracle takes the mean over its own batch
        part = OR.logit_priors(x64) * w
        (d64,) = torch.autograd.grad(part, x64, cot.double())
        pri64 += part.detach()
        b_d.add(d[s], d64, where=_where(s))
        del x64, part, d64
    for i, n in enumerate(("kl", "kl_improper_gmrf", "kl_tv")):
        err, atol = abs(float(pri[i].detach()) - float(pri64[i])), own_error_atol(pri32[i], pri64[i])
        assert err <= atol + RTOL * abs(float(pri64[i])), f"{n}: {float(pri[i].detach())!r} vs float64 {float(pri64[i])!r}"
    b_d.check()


# ------------------------------------------------------------------------------------------------ weak cross entropy
@pytest.mark.parametrize("mode", ["cross_entropy", "entropy"])
@pytest.mark.parametrize("name", list(CASES))
def test_weak_cross_entropy(ups, name, mode):
    c = CASES[name]
    K = c["K"]
    x = _place(_logits(c, 10), c["misaligned"]).requires_grad_(True)
    n_pix = x.numel() // K
    v = ups.model.weak_cross_entropy(x, mode)
    cot = 0.9 * n_pix                                                # keeps the gradient entries O(1)
    (d,) = torch.autograd.grad(v, x, torch.tensor(cot, device="cuda"))
    v32 = OR.weak_cross_entropy(x.detach(), mode)
    torch.cuda.synchronize()
    g = cot / n_pix
    total64 = 0.0
    b_d = _Bound(f"d logits ({mode})")
    for s in _chunks(c):
        xc = x[s].detach()
        lsm = torch.log_softmax(xc.double(), -1)
        p64 = lsm.exp()
        if mode == "cross_entropy":
            p32 = OP.softmax(xc)       # canonical: the kernels' probabilities, hence their hard labels
            lab = (p32 == p32.amax(-1, keepdim=True)).double()
            del p32
        else:
            lab = p64
        total64 += float(-(lab * lsm).sum())
        dot = (p64 * lsm).sum(-1, keepdim=True)
        b_d.add(d[s], g * ((p64 - lab) - p64 * (lsm - dot)), where=_where(s))
        del lsm, p64, lab, dot
    v64 = total64 / n_pix
    err, atol = abs(float(v.detach()) - v64), own_error_atol(v32, torch.tensor(v64))
    assert err <= atol + RTOL * abs(v64), f"{mode}: {float(v.detach())!r} vs float64 {v64!r}: |d| {err:.3e} > {atol:.3e} + rtol"
    b_d.check()


# ------------------------------------------------------------------------------------------------ spatial softmax
@pytest.mark.parametrize("name", list(CASES))
def test_spatial_softmax(ups, name):
    """Softmax over H*W for every (sample, part).  The probabilities are about 1/P, so 1e-5 absolute would accept
    anything: they are held to 1e-4 relative, with 1e-37 absolute for fp32 underflow.  dx = p (g - sum p g): the 1e-5
    absolute tolerance applies to the factor g - sum p g."""
    c = CASES[name]
    B, S, K = c["B"], c["S"], c["K"]
    P = S * S
    x = _place(_logits(c, 11), c["misaligned"]).requires_grad_(True)
    pr = ups.nn.spatial_softmax(x)
    gy = torch.randn(x.shape, device="cuda", generator=_gen(12))
    (dx,) = torch.autograd.grad(pr, x, gy)
    torch.cuda.synchronize()
    b_p, b_dx = _Bound("spatial softmax"), _Bound("d spatial softmax")
    for s in _chunks(c):
        n = s.stop - s.start
        p64 = torch.softmax(x[s].detach().double().view(n, P, K), 1)
        b_p.add(pr[s].view(n, P, K), p64, where=_where(s), atol=1e-37)
        g64 = gy[s].double().view(n, P, K)
        b_dx.add(dx[s].view(n, P, K), p64 * (g64 - (p64 * g64).sum(1, keepdim=True)), where=_where(s),
                 atol=ATOL * p64 + 1e-37)
        del p64, g64
    b_p.check()
    b_dx.check()


# ------------------------------------------------------------------------------------------------ mean-field sampling
@pytest.mark.parametrize("name", list(CASES))
def test_mean_field_sample_and_softmax(ups, name):
    c = CASES[name]
    K = c["K"]
    noise = 0.7
    x = _place(_logits(c, 13), c["misaligned"])
    eps = torch.randn(x.shape, device="cuda", generator=_gen(14))
    dist = ups.nn.MeanFieldDistribution(x, K)
    smp = None if c["misaligned"] else dist.sample(noise, eps=eps)
    lg, pr, labels, hard = dist.sample_softmax(noise, eps=eps)
    torch.cuda.synchronize()
    for s in _chunks(c):
        w = _where(s)
        want = _oracle(lambda m, e: OR.mean_field_sample(m, e, noise), x[s], eps[s])
        if smp is not None:
            _same_bits(smp[s], want, f"sample (samples {w})")
        _same_bits(lg[s], want, f"sampled logits (samples {w})")
        p_o = _oracle(OP.softmax, want)
        _same_bits(pr[s], p_o, f"probs (samples {w})")
        _same_bits(hard[s], _oracle(lambda p: OP.straight_through_estimator(OP.hard_max(p, 3), p), p_o),
                   f"hard mask (samples {w})")
        assert labels.dtype == torch.int64 and torch.equal(labels[s], OP.argmax_labels(p_o)), f"labels (samples {w})"
        del want, p_o


# ------------------------------------------------------------------------------------------------ mask2rgb
@pytest.mark.parametrize("name", list(CASES))
def test_mask2rgb(ups, name):
    c = CASES[name]
    K = c["K"]
    p = _place(torch.softmax(_logits(c, 15), -1), c["misaligned"])   # the all-equal rows tie: first maximum
    colors = torch.rand(K, 3, generator=torch.Generator().manual_seed(16))
    hot = ups.nn.mask2rgb(p, True, colors=colors)
    soft = ups.nn.mask2rgb(p, False, colors=colors)
    torch.cuda.synchronize()
    table64 = ((colors.double() - 0.5) * 2).float().double().cuda()
    b_soft = _Bound("mask2rgb soft")
    for s in _chunks(c):
        want = _oracle(lambda m: OR.mask2rgb(m, colors.to(m.device), True), p[s])
        _same_bits(hot[s], want, f"mask2rgb hot (samples {_where(s)})")
        b_soft.add(soft[s], torch.einsum("bhwk,kc->bhwc", p[s].double(), table64), where=_where(s))
        del want
    b_soft.check()
