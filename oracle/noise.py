"""TEST INFRASTRUCTURE — the mean-field logit noise the kernels draw (csrc/canon_math.cuh, "the mean-field logit noise"),
restated exactly: Philox4x32-10 in numpy uint64 arithmetic, then the canonical float operations of oracle/canon.py.

MeanFieldDistribution.sample (cub/code/nn.py:1421-1427) draws mean + noise_level * N(0,1).  TF's RNG stream cannot be
reproduced; the project's draw is a counter-based one, a pure function of (seed, draw, global pixel, part), so that the
kernels generate it in registers and this file restates it bit for bit.
"""
import numpy as np
import torch

from . import priors as PR
from . import step as OS
from .canon import _f32, log_canon

_PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
_PHILOX_W = (np.uint64(0x9E3779B9), np.uint64(0xBB67AE85))
_U32 = np.uint64(0xFFFFFFFF)
_PIO2 = 1.57079632679489662
_SIN_P = (-1.9515295891e-4, 8.3321608736e-3, -1.6666654611e-1)
_COS_P = (2.443315711809948e-5, -1.388731625493765e-3, 4.166664568298827e-2)


def philox4x32_10(ctr: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x32-10 (Random123 constants).  ctr [..., 4], key [..., 2] uint32 -> [..., 4] uint32, exact integer
    arithmetic in uint64.  Round: (hi0, lo0) = M0*c0, (hi1, lo1) = M1*c2; c = (hi1^c1^k0, lo1, hi0^c3^k1, lo0);
    then key += (W0, W1)."""
    c = [np.asarray(ctr)[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = (np.asarray(key)[..., i].astype(np.uint64) for i in range(2))
    s32 = np.uint64(32)
    for _ in range(10):
        p0 = _PHILOX_M[0] * c[0]
        p1 = _PHILOX_M[1] * c[2]
        c = [(p1 >> s32) ^ c[1] ^ k0, p1 & _U32, (p0 >> s32) ^ c[3] ^ k1, p0 & _U32]
        k0 = (k0 + _PHILOX_W[0]) & _U32
        k1 = (k1 + _PHILOX_W[1]) & _U32
    return np.stack(c, -1).astype(np.uint32)


def uniform24(x: np.ndarray) -> torch.Tensor:
    """u = ((x >> 8) + 1) * 2^-24 in (0, 1]: exact in fp32."""
    n = ((np.asarray(x, dtype=np.uint32) >> np.uint32(8)) + np.uint32(1)).astype(np.float32)
    return torch.from_numpy(n) * _f32(2.0 ** -24)


def sincos2pi_canon(u: torch.Tensor):
    """(sin, cos) of 2*pi*u for u in [0, 1], canonical fp32 order:
        t = 4u;  q = floor(t);  f = t - q                  (exact)
        fold = f > 0.5;  g = fold ? 1 - f : f;  x = g * PIO2;  z = x*x
        sn = ((S0*z + S1)*z + S2);  sn = (sn*z)*x;  sn = sn + x
        cs = ((C0*z + C1)*z + C2);  cs = (cs*z)*z;  cs = cs - 0.5*z;  cs = cs + 1
        (s, c) = fold ? (cs, sn) : (sn, cs)                 sin, cos of (pi/2) f
        quadrant q mod 4:  0 (s, c)   1 (c, -s)   2 (-s, -c)   3 (-c, s)
    """
    assert u.dtype == torch.float32
    t = u * _f32(4.0)
    q = torch.floor(t)
    f = t - q
    fold = f > _f32(0.5)
    g = torch.where(fold, _f32(1.0) - f, f)
    x = g * _f32(_PIO2)
    z = x * x
    sn = _f32(_SIN_P[0]) * z + _f32(_SIN_P[1])
    sn = sn * z + _f32(_SIN_P[2])
    sn = (sn * z) * x
    sn = sn + x
    cs = _f32(_COS_P[0]) * z + _f32(_COS_P[1])
    cs = cs * z + _f32(_COS_P[2])
    cs = (cs * z) * z
    cs = cs - _f32(0.5) * z
    cs = cs + _f32(1.0)
    s, c = torch.where(fold, cs, sn), torch.where(fold, sn, cs)
    quad = q.to(torch.int32) & 3
    sin = torch.where(quad == 0, s, torch.where(quad == 1, c, torch.where(quad == 2, -s, -c)))
    cos = torch.where(quad == 0, c, torch.where(quad == 1, -s, torch.where(quad == 2, -c, s)))
    return sin, cos


def box_muller_canon(xa: np.ndarray, xb: np.ndarray):
    """r = sqrt(-2 * log_canon(u(xa)));  (r * cos(2 pi u(xb)), r * sin(2 pi u(xb)))  (IEEE sqrt, correctly rounded)."""
    lg = log_canon(uniform24(xa))
    r = torch.from_numpy(np.sqrt((_f32(-2.0) * lg).numpy()))
    s, c = sincos2pi_canon(uniform24(xb))
    return r * c, r * s


def normal_philox(seed: int, draw: int, pix_offset: int, n_pix: int, K: int) -> torch.Tensor:
    """eps [n_pix, K] fp32: the N(0,1) draw of global pixels pix_offset .. pix_offset + n_pix - 1 (what
    ups_normal_philox_fwd writes).  Part k of pixel g comes from Philox4x32-10 with counter (g lo, g hi, k // 4, draw)
    and key (seed lo, seed hi): parts 4j, 4j+1 from words (x0, x1), parts 4j+2, 4j+3 from (x2, x3)."""
    seed = int(seed)
    assert 0 <= seed < 2 ** 64 and draw >= 0 and pix_offset >= 0
    J = (K + 3) // 4
    g = np.arange(n_pix, dtype=np.uint64) + np.uint64(pix_offset)
    ctr = np.empty((n_pix, J, 4), np.uint32)
    ctr[..., 0] = (g & _U32).astype(np.uint32)[:, None]
    ctr[..., 1] = (g >> np.uint64(32)).astype(np.uint32)[:, None]
    ctr[..., 2] = np.arange(J, dtype=np.uint32)[None, :]
    ctr[..., 3] = np.uint32(draw)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32)
    x = philox4x32_10(ctr, key)
    z0, z1 = box_muller_canon(x[..., 0], x[..., 1])
    z2, z3 = box_muller_canon(x[..., 2], x[..., 3])
    return torch.stack([z0, z1, z2, z3], -1).reshape(n_pix, 4 * J)[:, :K].contiguous()


def sample_logits(mean, seed, draw, noise_level=1.0, sample_offset=0):
    """MeanFieldDistribution.sample with this draw: fl(mean + fl(noise_level * eps)), eps of global pixels
    (sample_offset + b) * S*S + p."""
    B, H, W, K = mean.shape
    eps = normal_philox(seed, draw, sample_offset * H * W, B * H * W, K).reshape(B, H, W, K)
    return PR.mean_field_sample(mean, eps, noise_level)


def step_forward_backward(views, coord, t_vector, l0, l1, feat, cot, seed, noise_level=1.0, sample_offset=0, **kw):
    """The chained step oracle (oracle/step.py) on the training step's sampled logits: l0, l1 are the means, sampled with
    draw 0 / 1.  d l / d mean is the identity, so the returned dl0, dl1 are the gradients of the means."""
    s0 = sample_logits(l0, seed, 0, noise_level, sample_offset)
    s1 = sample_logits(l1, seed, 1, noise_level, sample_offset)
    return OS.step_forward_backward(views, coord, t_vector, s0, s1, feat, cot, **kw)
