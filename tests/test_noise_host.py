"""CPU tier: the mean-field logit noise (csrc/canon_math.cuh, "the mean-field logit noise") in the host build of the header
the kernels compile, against oracle/ON.py bit for bit, against Random123's known answers, and as a N(0,1) sample."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import noise as ON, parts as P, priors as PR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "unsupervised-part-segmentation_b200", "csrc")
SIN_COS_BOUND = 1.2e-7       # |canonical - float64| of sin / cos(2 pi u) over every u = n * 2^-24 (measured: 9.1e-8)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("canon_host") / "libups_canon_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(CSRC, "canon_host.cpp"),
                           "-o", so])
    return ctypes.CDLL(so)


def fp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def host_normal(lib, seed, draw, pix_offset, n_pix, K):
    out = np.empty((n_pix, K), np.float32)
    lib.ups_host_normal_philox(ctypes.c_ulonglong(seed), ctypes.c_int(draw), ctypes.c_longlong(pix_offset),
                               ctypes.c_longlong(n_pix), ctypes.c_int(K), fp(out))
    return out


def bits(a):
    return np.ascontiguousarray(a).view(np.int32)


KNOWN = [  # Random123 kat_vectors, philox4x32_10: (counter, key, result)
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def test_philox_known_answers(lib):
    ctr = np.array([c for c, _, _ in KNOWN], np.uint32)
    key = np.array([k for _, k, _ in KNOWN], np.uint32)
    want = np.array([r for _, _, r in KNOWN], np.uint32)
    out = np.empty_like(ctr)
    lib.ups_host_philox(fp(ctr), fp(key), fp(out), ctypes.c_longlong(len(KNOWN)))
    assert np.array_equal(out, want)
    assert np.array_equal(ON.philox4x32_10(ctr, key), want)


@pytest.mark.parametrize("seed,draw,pix_offset,n_pix,K", [
    (0, 0, 0, 62_500, 16),                              # 1e6 draws
    (0x0123456789ABCDEF, 1, 2 ** 32 - 20_000, 40_000, 25),  # global pixel indices cross 2^32 (counter word 1)
    (2 ** 64 - 1, 0, 2 ** 40 + 7, 20_000, 3),
    (977, 1, 5, 10_000, 64),
])
def test_host_draw_equals_oracle(lib, seed, draw, pix_offset, n_pix, K):
    out = host_normal(lib, seed, draw, pix_offset, n_pix, K)
    ref = ON.normal_philox(seed, draw, pix_offset, n_pix, K).numpy()
    assert np.array_equal(bits(out), bits(ref))
    assert np.isfinite(out).all() and np.abs(out).max() <= 5.77


def test_box_muller_edges_equal_oracle(lib):
    """u = 1 (x >> 8 all ones: log 1 = 0, r = -0) and u = 2^-24 (x < 256: the largest radius), every quadrant of u_b."""
    g = np.random.default_rng(0)
    xa = np.concatenate([np.full(8, 0xFFFFFFFF), np.zeros(8), np.full(8, 255), g.integers(0, 2 ** 32, 100_000)])
    xb = np.concatenate([np.array([0, 0x3FFFFF00, 0x40000000, 0x7FFFFF00, 0x80000000, 0xBFFFFF00, 0xC0000000, 0xFFFFFFFF])] * 3 +
                        [g.integers(0, 2 ** 32, 100_000)])
    xa, xb = xa.astype(np.uint32), xb.astype(np.uint32)
    za, zb = np.empty(xa.size, np.float32), np.empty(xa.size, np.float32)
    lib.ups_host_box_muller(fp(xa), fp(xb), fp(za), fp(zb), ctypes.c_longlong(xa.size))
    ra, rb = ON.box_muller_canon(xa, xb)
    assert np.array_equal(bits(za), bits(ra.numpy())) and np.array_equal(bits(zb), bits(rb.numpy()))
    assert not za[:8].any() and not zb[:8].any()
    r_max = np.sqrt(-2 * np.log(2.0 ** -24))
    assert np.abs(np.hypot(za[8:16].astype(np.float64), zb[8:16]) - r_max).max() < 1e-5
    assert np.isfinite(za).all() and np.isfinite(zb).all()


def test_sin_cos_over_the_whole_quadrant_grid(lib):
    """Every uniform the draw can produce, u = n * 2^-24, n = 1 .. 2^24: host == oracle bit for bit, and within
    SIN_COS_BOUND of float64."""
    u = (np.arange(1, 2 ** 24 + 1, dtype=np.float64) * 2.0 ** -24).astype(np.float32)
    s, c = np.empty_like(u), np.empty_like(u)
    lib.ups_host_sincos2pi(fp(u), fp(s), fp(c), ctypes.c_longlong(u.size))
    so, co = ON.sincos2pi_canon(torch.from_numpy(u))
    assert np.array_equal(bits(s), bits(so.numpy())) and np.array_equal(bits(c), bits(co.numpy()))
    a = 2 * np.pi * u.astype(np.float64)
    assert np.abs(s - np.sin(a)).max() <= SIN_COS_BOUND
    assert np.abs(c - np.cos(a)).max() <= SIN_COS_BOUND
    assert s[-1] == 0.0 and c[-1] == 1.0                     # u = 1: angle 2 pi


def test_draw_does_not_depend_on_k_or_batch_split(lib):
    seed = 31337
    a = host_normal(lib, seed, 0, 0, 4096, 25)
    b = host_normal(lib, seed, 0, 0, 4096, 32)
    assert np.array_equal(bits(a), bits(b[:, :25]))
    whole = host_normal(lib, seed, 1, 0, 2 * 4096, 16)
    halves = np.concatenate([host_normal(lib, seed, 1, 0, 4096, 16), host_normal(lib, seed, 1, 4096, 4096, 16)])
    assert np.array_equal(bits(whole), bits(halves))
    assert not np.array_equal(bits(host_normal(lib, seed, 0, 0, 4096, 16)), bits(whole[:4096]))   # draw 0 != draw 1
    assert not np.array_equal(bits(host_normal(lib, seed + 1, 1, 0, 4096, 16)), bits(whole[:4096]))


def test_padding_and_zero_noise_level():
    """-inf (a padded part) + noise stays -inf; noise_level = 0 gives the noise-free probabilities, masks and labels."""
    g = torch.Generator().manual_seed(3)
    mean = torch.randn(2048, 25, generator=g) * 3
    mean[:64] = torch.round(mean[:64])
    eps = ON.normal_philox(5, 0, 0, 2048, 32)
    padded = torch.full((2048, 32), float("-inf"))
    padded[:, :25] = mean
    s = PR.mean_field_sample(padded, eps, 0.7)
    assert bool(torch.isneginf(s[:, 25:]).all()) and bool(torch.isfinite(s[:, :25]).all())
    assert torch.equal(P.softmax(s)[:, :25], P.softmax(s[:, :25]))
    z = PR.mean_field_sample(mean, eps[:, :25], 0.0)
    assert torch.equal(z, mean)
    pz, pm = P.softmax(z), P.softmax(mean)
    assert torch.equal(pz, pm) and torch.equal(torch.argmax(pz, -1), torch.argmax(pm, -1))


def test_statistics_of_1e7_draws(lib):
    """Over 10^7 draws: Kolmogorov-Smirnov against N(0,1) does not reject at 1 %; mean, variance and the correlations
    between draw 0 and draw 1 and between neighbouring pixels lie within 5 sigma of 0, 1, 0."""
    from scipy import stats
    n_pix, K = 625_000, 16
    z0 = host_normal(lib, 20261020, 0, 3 * 2 ** 31, n_pix, K).astype(np.float64)
    z1 = host_normal(lib, 20261020, 1, 3 * 2 ** 31, n_pix, K).astype(np.float64)
    x = z0.ravel()
    n = x.size
    assert n == 10 ** 7
    assert stats.kstest(x, "norm").pvalue > 0.01
    assert abs(x.mean()) < 5 / np.sqrt(n)
    assert abs(x.var() - 1) < 5 * np.sqrt(2 / n)
    assert abs(np.corrcoef(x, z1.ravel())[0, 1]) < 5 / np.sqrt(n)
    assert abs(np.corrcoef(z0[:-1].ravel(), z0[1:].ravel())[0, 1]) < 5 / np.sqrt(n - K)
    assert abs(np.corrcoef(z0[:, 0::2].ravel(), z0[:, 1::2].ravel())[0, 1]) < 5 / np.sqrt(n // 2)   # the two of a pair


def test_data_parallel_step_draws_at_its_global_sample_offset(monkeypatch):
    """DataParallelPartStep on rank r of N builds its PartStep with sample_offset = r * per_gpu_batch, so the ranks draw
    what one GPU draws over the global batch (the construction stops right after PartStep: no GPU is needed)."""
    import ups_b200.dp as dp
    import ups_b200.step as st

    class Stop(Exception):
        pass

    seen = {}

    def fake_step(*a, **kw):
        seen.update(kw, batch=a[0])
        raise Stop

    monkeypatch.setattr(st, "PartStep", fake_step)
    monkeypatch.setattr(dp.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dp.dist, "get_world_size", lambda: 4)
    for rank in range(4):
        monkeypatch.setattr(dp.dist, "get_rank", lambda r=rank: r)
        with pytest.raises(Stop):
            dp.DataParallelPartStep(64, 128, 16, 64)
        assert seen["batch"] == 64 and seen["sample_offset"] == 64 * rank
