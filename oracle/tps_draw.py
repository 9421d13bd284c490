"""TEST INFRASTRUCTURE — the TPS parameters the kernels draw (csrc/canon_math.cuh, "the TPS parameters"), restated
exactly: Philox4x32-10 of oracle/noise.py, then single correctly rounded fp32 operations.

tps_parameters (transformations.py:17-39) draws its fields with tf.random_uniform in [lo, hi).  The project's draw is a
pure function of (seed, view v, global sample g):
    words x[4j .. 4j+3] = Philox4x32-10(counter = (g lo, g hi, j, 2 + v), key = (seed lo, seed hi)),  j = 0 .. 9
    u(x)    = (x >> 8) * 2^-24                 in [0, 1), exact in fp32
    U       = fl(lo + fl(u * w))               lo, w = hi - lo formed in double and rounded to fp32 once (draw_scalars)
    words 0 .. 15   coord [8,2] = fl(base + U(-0.2, 0.2))       16 .. 31  vector [8,2] = U(-tps_scal, tps_scal)
          32, 33    offset = U(-off_scal, off_scal)              34, 35    offset_2, the same range
          36, 37    t_scal = fl(U(scal (1 - scal_var), scal (1 + scal_var)) * rescal)
          38        t = fl(rot_turn * fl(2u - 1)) (a signed fraction of a turn), rot_turn = fl(rot_scal / (2 pi));
                    (s, c) = sincos2pi_canon(|t|), s negated when t < 0;  rot_mat = [[c, -s], [s, c]]
Draws 0 and 1 of the same seed are the logit noise (oracle/noise.py), so no TPS counter is ever a noise counter.
"""
import math

import numpy as np
import torch

from .noise import _U32, philox4x32_10, sincos2pi_canon
from .tps import AttrDict

DRAW_TPS_VIEW0 = 2
CALLS, WORDS = 10, 39
_BASE = np.array([[-0.5, -0.5], [0.5, -0.5], [-0.5, 0.5], [0.5, 0.5],
                  [0.2, -0.2], [-0.2, 0.2], [0.2, 0.2], [-0.2, -0.2]], np.float32)
SCALAR_NAMES = ("coord_lo", "coord_w", "vec_lo", "vec_w", "off_lo", "off_w", "scal_lo", "scal_w", "rescal", "rot_turn")


def draw_scalars(scal, tps_scal, rot_scal, off_scal, scal_var, rescal=1, augm_scal=None):
    """The ten fp32 scalars of the draw (SCALAR_NAMES order) from tps_parameters' keyword arguments."""
    if augm_scal is not None:
        rescal = augm_scal
    if not 0.0 <= rot_scal <= math.pi:
        raise ValueError(f"rot_scal must lie in [0, pi], got {rot_scal}")
    lo_hi = [(-0.2, 0.2), (-tps_scal, tps_scal), (-off_scal, off_scal), (scal * (1.0 - scal_var), scal * (1.0 + scal_var))]
    out = []
    for lo, hi in lo_hi:
        out += [float(lo), float(hi) - float(lo)]
    out += [float(rescal), float(rot_scal) * (1.0 / (2.0 * math.pi))]
    return np.array(out, np.float64).astype(np.float32)


def counters(view, g_offset, n):
    """The Philox counters [n, CALLS, 4] of view `view`, global samples g_offset .. g_offset + n - 1."""
    g = np.arange(n, dtype=np.uint64) + np.uint64(g_offset)
    ctr = np.empty((n, CALLS, 4), np.uint32)
    ctr[..., 0] = (g & _U32).astype(np.uint32)[:, None]
    ctr[..., 1] = (g >> np.uint64(32)).astype(np.uint32)[:, None]
    ctr[..., 2] = np.arange(CALLS, dtype=np.uint32)[None, :]
    ctr[..., 3] = np.uint32(DRAW_TPS_VIEW0 + view)
    return ctr


def words(seed, view, g_offset, n):
    """x [n, 39] uint32: the words of the draw."""
    seed = int(seed)
    assert 0 <= seed < 2 ** 64 and view in (0, 1) and g_offset >= 0
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32)
    return philox4x32_10(counters(view, g_offset, n), key).reshape(n, 4 * CALLS)[:, :WORDS]


def uniform(x):
    """u = (x >> 8) * 2^-24 in [0, 1): exact in fp32."""
    return torch.from_numpy((np.asarray(x, np.uint32) >> np.uint32(8)).astype(np.float32)) * np.float32(2.0 ** -24)


def _f(v):
    return torch.tensor(np.float32(v))


def rotation_turn(x, rot_turn):
    """t = fl(rot_turn * fl(2u - 1)), the signed fraction of a turn that the rotation word gives."""
    return _f(rot_turn) * (_f(2.0) * uniform(x) - _f(1.0))


def fields(x, s):
    """The fields of words x [n, 39] under draw_scalars s: dict(coord [n,8,2], vector [n,8,2], offset [n,1,2],
    offset_2 [n,1,2], t_scal [n,2], rot_mat [n,2,2]) fp32, the layouts of tps_parameters."""
    x = np.asarray(x, np.uint32)
    n = x.shape[0]
    s = dict(zip(SCALAR_NAMES, (np.float32(v) for v in s)))

    def U(w, lo, wd):
        return _f(s[lo]) + uniform(w) * _f(s[wd])

    coord = torch.from_numpy(_BASE.reshape(16)).expand(n, 16) + U(x[:, 0:16], "coord_lo", "coord_w")
    vector = U(x[:, 16:32], "vec_lo", "vec_w")
    offset = U(x[:, 32:34], "off_lo", "off_w")
    offset_2 = U(x[:, 34:36], "off_lo", "off_w")
    t_scal = U(x[:, 36:38], "scal_lo", "scal_w") * _f(s["rescal"])
    t = rotation_turn(x[:, 38], s["rot_turn"])
    sn, c = sincos2pi_canon(t.abs())
    sn = torch.where(t < 0, -sn, sn)
    rot_mat = torch.stack([c, -sn, sn, c], -1).reshape(n, 2, 2)
    return dict(coord=coord.reshape(n, 8, 2), vector=vector.reshape(n, 8, 2), offset=offset.reshape(n, 1, 2),
                offset_2=offset_2.reshape(n, 1, 2), t_scal=t_scal, rot_mat=rot_mat)


def tps_draw(seed, view, g_offset, n, s):
    """fields() of the draw of view `view`, global samples g_offset .. g_offset + n - 1."""
    return fields(words(seed, view, g_offset, n), s)


def tps_parameters(seed, n_per_view, views, sample_offset, **kw):
    """The rows [view 0 | view 1] (views = 2) or view 0 (views = 1) of samples sample_offset .. + n_per_view - 1: what
    ups_b200.tps.tps_parameters(views * n_per_view, seed=seed, sample_offset=sample_offset, views=views, **kw) returns."""
    s = draw_scalars(**kw)
    per = [tps_draw(seed, v, sample_offset, n_per_view, s) for v in range(views)]
    return AttrDict({k: torch.cat([p[k] for p in per], 0) for k in per[0]})
