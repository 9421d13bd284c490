"""CPU tier: the TPS parameters drawn from a seed (csrc/canon_math.cuh, "the TPS parameters") in the host build of the
header the kernels compile, against oracle/tps_draw.py bit for bit, as a sample of U(lo, hi), and for the properties the
device draw relies on (split invariance, counters apart from the logit noise's)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from oracle import noise as ON
from oracle import tps_draw as OD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "unsupervised-part-segmentation_b200", "csrc")
CUB_TPS = dict(scal=0.8, tps_scal=0.15, rot_scal=0.2, off_scal=0.2, scal_var=0.1, augm_scal=1.0)
PENN_TPS = dict(scal=0.95, tps_scal=0.08, rot_scal=0.05, off_scal=0.2, scal_var=0.05, augm_scal=1.0)
RANGES = [pytest.param(CUB_TPS, id="cub"), pytest.param(PENN_TPS, id="penn")]
SIN_COS_BOUND = 1.2e-7       # |sincos2pi_canon - float64| (tests/test_noise_host.py)
FIELDS = ("coord", "vector", "offset", "offset_2", "t_scal", "rot_mat")
SHAPES = dict(coord=(8, 2), vector=(8, 2), offset=(1, 2), offset_2=(1, 2), t_scal=(2,), rot_mat=(2, 2))


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("canon_host") / "libups_canon_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(CSRC, "canon_host.cpp"),
                           "-o", so])
    return ctypes.CDLL(so)


def fp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _out(n):
    return {k: np.empty((n,) + SHAPES[k], np.float32) for k in FIELDS}


def host_draw(lib, seed, view, g_offset, n, s):
    o = _out(n)
    lib.ups_host_tps_draw(ctypes.c_ulonglong(seed), ctypes.c_int(view), ctypes.c_ulonglong(g_offset), ctypes.c_longlong(n),
                          fp(np.ascontiguousarray(s, np.float32)), *[fp(o[k]) for k in FIELDS])
    return o


def host_fields(lib, x, s):
    x = np.ascontiguousarray(x, np.uint32)
    o = _out(x.shape[0])
    lib.ups_host_tps_fields(fp(x), fp(np.ascontiguousarray(s, np.float32)), *[fp(o[k]) for k in FIELDS],
                            ctypes.c_longlong(x.shape[0]))
    return o


def assert_same(h, o, what):
    for k in FIELDS:
        assert np.array_equal(bits(h[k]), bits(o[k].numpy())), f"{what}: {k}"


def extreme_words(n=4096, seed=0):
    """Words that give u = 0 (x >> 8 == 0) and u = 1 - 2^-24 (x >> 8 == 2^24 - 1) in every position, and mixtures."""
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, 256, (n, OD.WORDS), dtype=np.uint32)
    hi = (np.uint32(0xFFFFFF00) | lo).astype(np.uint32)
    pick = rng.integers(0, 3, (n, OD.WORDS))
    mixed = np.where(pick == 0, lo, np.where(pick == 1, hi, rng.integers(0, 2 ** 32, (n, OD.WORDS), dtype=np.uint32)))
    return np.concatenate([lo, hi, mixed.astype(np.uint32)])


@pytest.mark.parametrize("kw", RANGES)
def test_host_equals_oracle(lib, kw):
    """>= 10^5 samples per range: seeds near 0 and 2^64, g past 2^32, both views, and the extreme words."""
    s = OD.draw_scalars(**kw)
    n_total = 0
    for seed, view, g0, n in ((0, 0, 0, 30000), (2 ** 64 - 1, 1, 2 ** 32 - 7, 30000), (2 ** 64 - 12345, 0, 2 ** 40 + 3, 20000),
                              (0x5EED_0123_4567_89AB, 1, 17, 20000)):
        assert_same(host_draw(lib, seed, view, g0, n, s), OD.tps_draw(seed, view, g0, n, s), f"seed={seed} view={view}")
        n_total += n
    x = extreme_words()
    assert_same(host_fields(lib, x, s), OD.fields(x, s), "extreme words")
    assert n_total + x.shape[0] >= 10 ** 5


@pytest.mark.parametrize("kw", RANGES)
def test_scalars_match_the_package(kw):
    from ups_b200 import tps
    assert np.array_equal(np.array(tps.draw_scalars(**kw), np.float32).view(np.int32), OD.draw_scalars(**kw).view(np.int32))


def _ranges(kw, s):
    """field -> (lo, hi) of every element in double, from the fp32 scalars: U in [lo32, lo32 + w32), coord = fl(base + U)
    in [fl(base + lo32), base + lo32 + w32)."""
    d = dict(zip(OD.SCALAR_NAMES, (float(v) for v in s)))
    base = OD._BASE.astype(np.float64)
    coord_lo = (OD._BASE + np.float32(d["coord_lo"])).astype(np.float64)
    return dict(coord=(coord_lo, base + d["coord_lo"] + d["coord_w"]),
                vector=(d["vec_lo"], d["vec_lo"] + d["vec_w"]),
                offset=(d["off_lo"], d["off_lo"] + d["off_w"]), offset_2=(d["off_lo"], d["off_lo"] + d["off_w"]),
                t_scal=(d["scal_lo"] * d["rescal"], (d["scal_lo"] + d["scal_w"]) * d["rescal"]))


@pytest.mark.parametrize("kw", RANGES)
def test_fields_in_half_open_ranges(lib, kw):
    s = OD.draw_scalars(**kw)
    x = extreme_words()
    for o in (host_draw(lib, 99, 0, 0, 200000, s), host_draw(lib, 99, 1, 0, 200000, s), host_fields(lib, x, s)):
        for k, (lo, hi) in _ranges(kw, s).items():
            v = o[k].astype(np.float64)
            assert np.all(v >= lo) and np.all(v < hi), k
        # the angle within [-rot_scal, rot_scal]
        assert np.all(np.abs(o["rot_mat"][:, 1, 0]) <= math.sin(kw["rot_scal"]) + 1e-7)
    # u = 0 gives lo exactly, u = 1 - 2^-24 the largest value below hi
    o = host_fields(lib, np.zeros((1, OD.WORDS), np.uint32), s)
    d = dict(zip(OD.SCALAR_NAMES, s))
    assert o["vector"][0, 0, 0] == d["vec_lo"] and o["offset"][0, 0, 0] == d["off_lo"]
    t = OD.rotation_turn(np.array([0, 0xFFFFFFFF], np.uint32), d["rot_turn"]).numpy()
    assert t[0] == -d["rot_turn"] and t[1] < d["rot_turn"]


@pytest.mark.parametrize("kw", RANGES)
def test_each_field_is_uniform(lib, kw):
    """Kolmogorov-Smirnov of each of the 39 fields against U(lo, hi) over 10^6 samples (fixed seed)."""
    n = 10 ** 6
    o = host_draw(lib, 2024, 1, 10 ** 9, n, OD.draw_scalars(**kw))
    cols = []
    jitter = o["coord"].reshape(n, 16).astype(np.float64) - OD._BASE.reshape(16).astype(np.float64)
    cols += [(f"coord[{i}]", jitter[:, i], -0.2, 0.2) for i in range(16)]
    cols += [(f"vector[{i}]", o["vector"].reshape(n, 16)[:, i], -kw["tps_scal"], kw["tps_scal"]) for i in range(16)]
    for k in ("offset", "offset_2"):
        cols += [(f"{k}[{i}]", o[k].reshape(n, 2)[:, i], -kw["off_scal"], kw["off_scal"]) for i in range(2)]
    sl, sh = kw["scal"] * (1 - kw["scal_var"]) * kw["augm_scal"], kw["scal"] * (1 + kw["scal_var"]) * kw["augm_scal"]
    cols += [(f"t_scal[{i}]", o["t_scal"][:, i], sl, sh) for i in range(2)]
    angle = np.arctan2(o["rot_mat"][:, 1, 0].astype(np.float64), o["rot_mat"][:, 0, 0].astype(np.float64))
    cols.append(("angle", angle, -kw["rot_scal"], kw["rot_scal"]))
    assert len(cols) == OD.WORDS
    for name, v, lo, hi in cols:
        p = stats.kstest(np.asarray(v, np.float64), stats.uniform(loc=lo, scale=hi - lo).cdf).pvalue
        assert p > 1e-4, (name, p)


@pytest.mark.parametrize("rot_scal", [0.2, 0.05, 1.0, math.pi])
def test_rotation_accuracy(lib, rot_scal):
    """rot_mat against float64 cos / sin of the angle rot_scal (2u - 1) the word stands for: within the canonical
    sin / cos bound plus 2^-23 |angle| (the two fp32 roundings of the turn)."""
    kw = dict(CUB_TPS, rot_scal=rot_scal)
    s = OD.draw_scalars(**kw)
    n = 200000
    seed, view, g0 = 77, 0, 5
    o = host_draw(lib, seed, view, g0, n, s)
    u = (OD.words(seed, view, g0, n)[:, 38] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    theta = rot_scal * (2.0 * u - 1.0)
    bound = SIN_COS_BOUND + np.abs(theta) * 2.0 ** -23
    r = o["rot_mat"].astype(np.float64)
    c, sn = np.cos(theta), np.sin(theta)
    for got, want in ((r[:, 0, 0], c), (r[:, 1, 1], c), (r[:, 1, 0], sn), (r[:, 0, 1], -sn)):
        assert np.all(np.abs(got - want) <= bound), np.max(np.abs(got - want) - bound)


def test_rot_scal_outside_half_turn_raises():
    with pytest.raises(ValueError, match="rot_scal"):
        OD.draw_scalars(**dict(CUB_TPS, rot_scal=math.pi + 1e-6))
    with pytest.raises(ValueError, match="rot_scal"):
        OD.draw_scalars(**dict(CUB_TPS, rot_scal=-0.1))


@pytest.mark.parametrize("view", [0, 1])
def test_split_invariance(lib, view):
    """The draws of samples [0, 2n) equal those of [0, n) followed by [n, 2n): the draw does not depend on the split."""
    s = OD.draw_scalars(**CUB_TPS)
    n = 3001
    whole = host_draw(lib, 31337, view, 0, 2 * n, s)
    a, b = host_draw(lib, 31337, view, 0, n, s), host_draw(lib, 31337, view, n, n, s)
    for k in FIELDS:
        assert np.array_equal(bits(whole[k]), bits(np.concatenate([a[k], b[k]]))), k


def test_counters_apart_from_the_logit_noise():
    """Under one seed, no TPS counter (draws 2, 3) is a counter of the logit noise (draws 0, 1), even where the global
    sample index of one equals the global pixel index of the other."""
    n = 4096
    tps = np.concatenate([OD.counters(v, 0, n) for v in (0, 1)]).reshape(-1, 4)
    assert set(np.unique(tps[:, 3]).tolist()) == {2, 3}
    g = np.arange(n, dtype=np.uint64)
    J = 7                                      # K = 25: parts 4j .. 4j + 3 for j < 7
    noise = np.empty((2, n, J, 4), np.uint32)  # oracle/noise.py::normal_philox's counters
    noise[..., 0] = (g & ON._U32).astype(np.uint32)[None, :, None]
    noise[..., 1] = (g >> np.uint64(32)).astype(np.uint32)[None, :, None]
    noise[..., 2] = np.arange(J, dtype=np.uint32)[None, None, :]
    noise[..., 3] = np.arange(2, dtype=np.uint32)[:, None, None]
    as_set = lambda c: set(map(tuple, c.reshape(-1, 4).tolist()))
    assert not as_set(tps) & as_set(noise)
    # and the words are Philox of exactly those counters
    key = np.array([0x89AB, 0x5EED], np.uint32)
    x = ON.philox4x32_10(OD.counters(1, 0, 8), key).reshape(8, 40)[:, :OD.WORDS]
    assert np.array_equal(x, OD.words((0x5EED << 32) | 0x89AB, 1, 0, 8))
