"""PyTorch custom operators `ups::*` over the C ABI (include/ups_b200.h).

PyTorch is plumbing here: it owns device memory and streams and records the autograd graph;
every numeric result comes from the sm_100a kernels in csrc/.  There is no CPU
implementation: a CPU tensor raises.
"""
import math
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _cabi as C
from .step import decode_bwd_tc_ok, kernel_route


def _stream(t: Tensor):
    """The current stream of the device that owns `t`, tagged with that device: C.call makes the device current
    for the duration of the call (the C ABI launches on the calling thread's current device)."""
    return C.StreamHandle(torch.cuda.current_stream(t.device).cuda_stream, t.device.index)


def _f32(t: Tensor, name="tensor") -> Tensor:
    if not t.is_cuda:
        raise C.UpsError(f"ups_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if t.dtype != torch.float32:
        raise C.UpsError(f"ups_b200: {name} must be float32, got {t.dtype}")
    return t.contiguous()


def _ptr(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _ws(nbytes: int, like: Tensor) -> Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=like.device)


def _op(name, schema_fn, fake_fn, backward=None, setup=None):
    op = torch.library.custom_op(f"ups::{name}", mutates_args=())(schema_fn)
    op.register_fake(fake_fn)
    if backward is not None:
        op.register_autograd(backward, setup_context=setup)
    return op


# ------------------------------------------------------------------ image ingest
def _views_u8_to_f32(images: Tensor) -> Tensor:
    if not images.is_cuda:
        raise C.UpsError("ups_b200: images must be a CUDA tensor (no CPU fallback exists)")
    if images.dtype != torch.uint8:
        raise C.UpsError(f"ups_b200: images must be uint8, got {images.dtype}")
    images = images.contiguous()
    out = torch.empty(images.shape, dtype=torch.float32, device=images.device)
    C.call("ups_views_u8_to_f32", images.data_ptr(), out.data_ptr(), images.numel(), _stream(images))
    return out


views_u8_to_f32 = _op("views_u8_to_f32", _views_u8_to_f32,
                      lambda images: torch.empty(images.shape, dtype=torch.float32, device=images.device))


# ------------------------------------------------------------------ TPS
def _tps_input_param(coord: Tensor, vector: Tensor, offset: Tensor, offset_2: Tensor, t_scal: Tensor,
                     rot_mat: Tensor) -> Tensor:
    a = [_f32(t) for t in (coord, vector, offset, offset_2, t_scal, rot_mat)]
    N = a[0].shape[0]
    out = torch.empty_like(a[0])
    C.call("ups_tps_input_param", *[t.data_ptr() for t in a], out.data_ptr(), N, _stream(out))
    return out


tps_input_param = _op("tps_input_param", _tps_input_param, lambda c, v, o, o2, s, r: torch.empty_like(c))


def _tps_solve(coord: Tensor, vector: Tensor) -> Tensor:
    coord, vector = _f32(coord), _f32(vector)
    N = coord.shape[0]
    T = torch.empty(N, 2, 11, dtype=torch.float32, device=coord.device)
    C.call("ups_tps_solve", coord.data_ptr(), vector.data_ptr(), T.data_ptr(), N, _stream(coord))
    return T


tps_solve = _op("tps_solve", _tps_solve, lambda c, v: c.new_empty(c.shape[0], 2, 11))


def _tps_warp(U: Tensor, coord: Tensor, T: Tensor, out_size: int, move: Optional[Tensor],
              scal: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    U, coord, T = _f32(U, "U"), _f32(coord, "coord"), _f32(T, "T")
    move = None if move is None else _f32(move, "move")
    scal = None if scal is None else _f32(scal, "scal")
    N, H, W, Cc = U.shape
    out = torch.empty(N, out_size, out_size, Cc, dtype=torch.float32, device=U.device)
    mesh = torch.empty(N, out_size, out_size, 2, dtype=torch.float32, device=U.device)
    C.call("ups_tps_warp_fwd", U.data_ptr(), coord.data_ptr(), T.data_ptr(), _ptr(move), _ptr(scal),
           out.data_ptr(), mesh.data_ptr(), N, H, W, Cc, out_size, out_size, _stream(U))
    return out, mesh


def _tps_warp_fake(U, coord, T, out_size, move, scal):
    N, H, W, Cc = U.shape
    return U.new_empty(N, out_size, out_size, Cc), U.new_empty(N, out_size, out_size, 2)


def _tps_warp_setup(ctx, inputs, output):
    U, coord, T, out_size, move, scal = inputs
    # gradients reach the images only: the reference draws the TPS / crop parameters at random (model.py:298-300) and
    # they are data, not variables.  Asking for more raises instead of silently returning nothing (ADVICE r1).
    ctx.set_materialize_grads(False)
    ctx.param_grad = any(t is not None and t.requires_grad for t in (coord, T, move, scal))
    ctx.save_for_backward(coord, T, *([move, scal] if move is not None else []))
    ctx.has_move = move is not None
    ctx.shape = tuple(U.shape)
    ctx.out_size = out_size


def _tps_warp_bwd(ctx, g_out, g_mesh):
    if ctx.param_grad:
        raise C.UpsError("ups_b200: ThinPlateSpline has no gradient with respect to coord / T / move / scal "
                         "(the warp parameters are data in the reference, model.py:298-300); detach them")
    if g_mesh is not None:
        raise C.UpsError("ups_b200: no gradient flows through the sampling mesh (t_arr) of ThinPlateSpline")
    saved = ctx.saved_tensors
    if g_out is None:
        return None, None, None, None, None, None
    coord, T = saved[0], saved[1]
    move, scal = (saved[2], saved[3]) if ctx.has_move else (None, None)
    dU = tps_warp_grad(g_out, coord, T, list(ctx.shape), ctx.out_size, move, scal)
    return dU, None, None, None, None, None


def _tps_warp_grad(g_out: Tensor, coord: Tensor, T: Tensor, shape: list[int], out_size: int,
                   move: Optional[Tensor], scal: Optional[Tensor]) -> Tensor:
    g_out = _f32(g_out, "g_out")
    N, H, W, Cc = shape
    dU = torch.empty(N, H, W, Cc, dtype=torch.float32, device=g_out.device)
    C.call("ups_tps_warp_bwd", g_out.data_ptr(), coord.data_ptr(), T.data_ptr(), _ptr(move), _ptr(scal),
           dU.data_ptr(), N, H, W, Cc, out_size, out_size, _stream(g_out))
    return dU


tps_warp_grad = _op("tps_warp_grad", _tps_warp_grad,
                    lambda g, c, T, shape, o, m, s: g.new_empty(shape))
tps_warp = _op("tps_warp", _tps_warp, _tps_warp_fake, _tps_warp_bwd, _tps_warp_setup)


# ------------------------------------------------------------------ softmax family
def _part_softmax_full(logits: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    x = _f32(logits, "logits")
    K = x.shape[-1]
    n_pix = x.numel() // K
    probs = torch.empty_like(x)
    hard = torch.empty_like(x)
    labels = torch.empty(x.shape[:-1], dtype=torch.int64, device=x.device)
    C.call("ups_part_softmax_fwd", x.data_ptr(), probs.data_ptr(), labels.data_ptr(), hard.data_ptr(), n_pix, K,
           _stream(x))
    return probs, labels, hard


def _part_softmax(logits: Tensor) -> Tensor:
    x = _f32(logits, "logits")
    K = x.shape[-1]
    probs = torch.empty_like(x)
    C.call("ups_part_softmax_fwd", x.data_ptr(), probs.data_ptr(), None, None, x.numel() // K, K, _stream(x))
    return probs


def _part_softmax_grad(probs: Tensor, g: Tensor) -> Tensor:
    probs, g = _f32(probs), _f32(g)
    K = probs.shape[-1]
    dx = torch.empty_like(probs)
    C.call("ups_part_softmax_bwd", probs.data_ptr(), g.data_ptr(), dx.data_ptr(), probs.numel() // K, K, _stream(probs))
    return dx


part_softmax_grad = _op("part_softmax_grad", _part_softmax_grad, lambda p, g: torch.empty_like(p))
part_softmax = _op("part_softmax", _part_softmax, lambda x: torch.empty_like(x),
                   lambda ctx, g: part_softmax_grad(ctx.saved_tensors[0], g),
                   lambda ctx, inputs, output: ctx.save_for_backward(output))


def _psf_bwd(ctx, g_probs, g_labels, g_hard):
    # straight-through: the hard mask passes its cotangent unchanged to the probabilities
    (p,) = ctx.saved_tensors
    g = g_probs if g_hard is None else (g_hard if g_probs is None else g_probs + g_hard)
    return part_softmax_grad(p, g)


part_softmax_full = _op(
    "part_softmax_full", _part_softmax_full,
    lambda x: (torch.empty_like(x), x.new_empty(x.shape[:-1], dtype=torch.int64), torch.empty_like(x)),
    _psf_bwd, lambda ctx, inputs, output: ctx.save_for_backward(output[0]))


def _spatial_softmax(x: Tensor) -> Tensor:
    x = _f32(x)
    N, H, W, Cc = x.shape
    out = torch.empty_like(x)
    C.call("ups_spatial_softmax_fwd", x.data_ptr(), out.data_ptr(), N, H * W, Cc, _stream(x))
    return out


def _spatial_softmax_grad(probs: Tensor, g: Tensor) -> Tensor:
    probs, g = _f32(probs), _f32(g)
    N, H, W, Cc = probs.shape
    dx = torch.empty_like(probs)
    C.call("ups_spatial_softmax_bwd", probs.data_ptr(), g.data_ptr(), dx.data_ptr(), N, H * W, Cc, _stream(probs))
    return dx


spatial_softmax_grad = _op("spatial_softmax_grad", _spatial_softmax_grad, lambda p, g: torch.empty_like(p))
spatial_softmax = _op("spatial_softmax", _spatial_softmax, lambda x: torch.empty_like(x),
                      lambda ctx, g: spatial_softmax_grad(ctx.saved_tensors[0], g),
                      lambda ctx, inputs, output: ctx.save_for_backward(output))


def _hard_max(y: Tensor) -> Tensor:
    y = _f32(y)
    K = y.shape[-1]
    out = torch.empty_like(y)
    C.call("ups_hard_max_fwd", y.data_ptr(), out.data_ptr(), y.numel() // K, K, _stream(y))
    return out


hard_max = _op("hard_max", _hard_max, lambda y: torch.empty_like(y))   # tf.equal: no gradient


def _straight_through(y_hard: Tensor, y: Tensor) -> Tensor:
    y_hard, y = _f32(y_hard), _f32(y)
    out = torch.empty_like(y)
    C.call("ups_straight_through_fwd", y_hard.data_ptr(), y.data_ptr(), out.data_ptr(), y.numel(), _stream(y_hard))
    return out


straight_through = _op("straight_through", _straight_through, lambda h, y: torch.empty_like(y),
                       lambda ctx, g: (None, g), lambda ctx, inputs, output: None)


def _argmax(y: Tensor) -> Tensor:
    y = _f32(y)
    K = y.shape[-1]
    out = torch.empty(y.shape[:-1], dtype=torch.int64, device=y.device)
    C.call("ups_argmax_fwd", y.data_ptr(), out.data_ptr(), y.numel() // K, K, _stream(y))
    return out


argmax = _op("argmax", _argmax, lambda y: y.new_empty(y.shape[:-1], dtype=torch.int64))


def _one_hot(labels: Tensor, depth: int) -> Tensor:
    labels = labels.contiguous()
    out = torch.empty(*labels.shape, depth, dtype=torch.float32, device=labels.device)
    C.call("ups_one_hot_fwd", labels.data_ptr(), out.data_ptr(), labels.numel(), depth, _stream(labels))
    return out


one_hot = _op("one_hot", _one_hot, lambda l, d: l.new_empty(*l.shape, d, dtype=torch.float32))


# ------------------------------------------------------------------ mask_parts / apply_partwise
def _dims_bpk(image: Tensor, mask: Tensor):
    B = image.shape[0]
    P = image.numel() // (B * image.shape[-1]) if B else 0
    return B, P, mask.shape[-1], image.shape[-1]


def _mask_parts(image: Tensor, mask: Tensor, part_major: bool) -> Tensor:
    image, mask = _f32(image, "image"), _f32(mask, "mask")
    B, P, K, Cc = _dims_bpk(image, mask)
    sp = image.shape[1:-1]
    out = torch.empty((K * B, *sp, Cc) if part_major else (B, *sp, K, Cc), dtype=torch.float32, device=image.device)
    C.call("ups_mask_parts_fwd", image.data_ptr(), mask.data_ptr(), out.data_ptr(), B, P, K, Cc, int(part_major),
           _stream(image))
    return out


def _mask_parts_fake(image, mask, part_major):
    B, K, Cc = image.shape[0], mask.shape[-1], image.shape[-1]
    sp = image.shape[1:-1]
    return image.new_empty((K * B, *sp, Cc) if part_major else (B, *sp, K, Cc))


def _mask_parts_grad(g: Tensor, image: Tensor, mask: Tensor, part_major: bool) -> Tuple[Tensor, Tensor]:
    g, image, mask = _f32(g), _f32(image), _f32(mask)
    B, P, K, Cc = _dims_bpk(image, mask)
    dimage, dmask = torch.empty_like(image), torch.empty_like(mask)
    C.call("ups_mask_parts_bwd", g.data_ptr(), image.data_ptr(), mask.data_ptr(), dimage.data_ptr(), dmask.data_ptr(),
           B, P, K, Cc, int(part_major), _stream(g))
    return dimage, dmask


mask_parts_grad = _op("mask_parts_grad", _mask_parts_grad,
                      lambda g, i, m, pm: (torch.empty_like(i), torch.empty_like(m)))


def _mask_parts_bwd(ctx, g):
    image, mask = ctx.saved_tensors
    di, dm = mask_parts_grad(g, image, mask, ctx.pm)
    return di, dm, None


def _mask_parts_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1])
    ctx.pm = inputs[2]


mask_parts = _op("mask_parts", _mask_parts, _mask_parts_fake, _mask_parts_bwd, _mask_parts_setup)


def _partwise_fold(x: Tensor) -> Tensor:
    x = _f32(x)
    B, K, Cc = x.shape[0], x.shape[-2], x.shape[-1]
    sp = x.shape[1:-2]
    P = x.numel() // (B * K * Cc) if B else 0
    y = torch.empty(K * B, *sp, Cc, dtype=torch.float32, device=x.device)
    C.call("ups_partwise_fold", x.data_ptr(), y.data_ptr(), B, P, K, Cc, _stream(x))
    return y


def _partwise_unfold(y: Tensor, parts: int) -> Tensor:
    y = _f32(y)
    KB, Cc = y.shape[0], y.shape[-1]
    B = KB // parts
    sp = y.shape[1:-1]
    P = y.numel() // (KB * Cc) if KB else 0
    x = torch.empty(B, *sp, parts, Cc, dtype=torch.float32, device=y.device)
    C.call("ups_partwise_unfold", y.data_ptr(), x.data_ptr(), B, P, parts, Cc, _stream(y))
    return x


partwise_fold = _op("partwise_fold", _partwise_fold,
                    lambda x: x.new_empty(x.shape[-2] * x.shape[0], *x.shape[1:-2], x.shape[-1]),
                    lambda ctx, g: partwise_unfold(g, ctx.parts),
                    lambda ctx, inputs, output: setattr(ctx, "parts", inputs[0].shape[-2]))
partwise_unfold = _op("partwise_unfold", _partwise_unfold,
                      lambda y, parts: y.new_empty(y.shape[0] // parts, *y.shape[1:-1], parts, y.shape[-1]),
                      lambda ctx, g: (partwise_fold(g), None), lambda ctx, inputs, output: None)


# ------------------------------------------------------------------ pooling
def _part_pool(fmap: Tensor, mask: Tensor, grouped: bool, scale: float) -> Tensor:
    fmap, mask = _f32(fmap, "feature_map"), _f32(mask, "mask")
    B, K, nf = fmap.shape[0], mask.shape[-1], fmap.shape[-1]
    P = mask.numel() // (B * K) if B else 0
    Fg = nf // K if grouped else nf
    out = torch.empty(B, K, Fg, dtype=torch.float32, device=fmap.device)
    ws = _ws(C.workspace_bytes(C.OP_POOL, B, P, K, Fg), fmap)
    C.call("ups_part_pool_fwd", fmap.data_ptr(), mask.data_ptr(), out.data_ptr(), B, P, K, Fg, int(grouped), scale,
           ws.data_ptr(), ws.numel(), _stream(fmap))
    return out


def _part_pool_fake(fmap, mask, grouped, scale):
    K = mask.shape[-1]
    return fmap.new_empty(fmap.shape[0], K, fmap.shape[-1] // K if grouped else fmap.shape[-1])


def _part_pool_grad(g: Tensor, fmap: Tensor, mask: Tensor, grouped: bool, scale: float) -> Tuple[Tensor, Tensor]:
    g, fmap, mask = _f32(g), _f32(fmap), _f32(mask)
    B, K, nf = fmap.shape[0], mask.shape[-1], fmap.shape[-1]
    P = mask.numel() // (B * K) if B else 0
    Fg = nf // K if grouped else nf
    dfmap, dmask = torch.empty_like(fmap), torch.empty_like(mask)
    C.call("ups_part_pool_bwd", g.data_ptr(), fmap.data_ptr(), mask.data_ptr(), dfmap.data_ptr(), dmask.data_ptr(),
           B, P, K, Fg, int(grouped), scale, _stream(g))
    return dfmap, dmask


part_pool_grad = _op("part_pool_grad", _part_pool_grad,
                     lambda g, f, m, gr, s: (torch.empty_like(f), torch.empty_like(m)))


def _part_pool_bwd(ctx, g):
    fmap, mask = ctx.saved_tensors
    df, dm = part_pool_grad(g, fmap, mask, ctx.grouped, ctx.scale)
    return df, dm, None, None


def _part_pool_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1])
    ctx.grouped, ctx.scale = inputs[2], inputs[3]


part_pool = _op("part_pool", _part_pool, _part_pool_fake, _part_pool_bwd, _part_pool_setup)


# ------------------------------------------------------------------ unpool / inject / gather
def _bpkf(feat: Tensor, mask: Tensor):
    B, K, F = feat.shape
    P = mask.numel() // (B * K) if B else 0
    return B, P, K, F


def _part_unpool(feat: Tensor, mask: Tensor) -> Tensor:
    feat, mask = _f32(feat, "feature_vectors"), _f32(mask, "mask")
    B, P, K, F = _bpkf(feat, mask)
    out = torch.empty(*mask.shape, F, dtype=torch.float32, device=feat.device)
    C.call("ups_part_unpool_fwd", feat.data_ptr(), mask.data_ptr(), out.data_ptr(), B, P, K, F, _stream(feat))
    return out


def _part_unpool_grad(g: Tensor, feat: Tensor, mask: Tensor) -> Tuple[Tensor, Tensor]:
    g, feat, mask = _f32(g), _f32(feat), _f32(mask)
    B, P, K, F = _bpkf(feat, mask)
    dfeat, dmask = torch.empty_like(feat), torch.empty_like(mask)
    ws = _ws(C.workspace_bytes(C.OP_POOL, B, P, K, F), feat)
    C.call("ups_part_unpool_bwd", g.data_ptr(), feat.data_ptr(), mask.data_ptr(), dfeat.data_ptr(), dmask.data_ptr(),
           B, P, K, F, ws.data_ptr(), ws.numel(), _stream(g))
    return dfeat, dmask


part_unpool_grad = _op("part_unpool_grad", _part_unpool_grad,
                       lambda g, f, m: (torch.empty_like(f), torch.empty_like(m)))
part_unpool = _op("part_unpool", _part_unpool, lambda f, m: m.new_empty(*m.shape, f.shape[-1]),
                  lambda ctx, g: part_unpool_grad(g, *ctx.saved_tensors),
                  lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1]))


def _part_inject(feat: Tensor, mask: Tensor) -> Tensor:
    feat, mask = _f32(feat, "feature_vectors"), _f32(mask, "mask")
    B, P, K, F = _bpkf(feat, mask)
    out = torch.empty(*mask.shape[:-1], F + K, dtype=torch.float32, device=feat.device)
    C.call("ups_part_inject_fwd", feat.data_ptr(), mask.data_ptr(), out.data_ptr(), B, P, K, F, _stream(feat))
    return out


def _part_inject_grad(g: Tensor, feat: Tensor, mask: Tensor) -> Tuple[Tensor, Tensor]:
    g, feat, mask = _f32(g), _f32(feat), _f32(mask)
    B, P, K, F = _bpkf(feat, mask)
    dfeat, dmask = torch.empty_like(feat), torch.empty_like(mask)
    ws = _ws(C.workspace_bytes(C.OP_INJECT_BWD, B, P, K, F), feat)
    C.call("ups_part_inject_bwd", g.data_ptr(), feat.data_ptr(), mask.data_ptr(), dfeat.data_ptr(), dmask.data_ptr(),
           B, P, K, F, ws.data_ptr(), ws.numel(), _stream(g))
    return dfeat, dmask


part_inject_grad = _op("part_inject_grad", _part_inject_grad,
                       lambda g, f, m: (torch.empty_like(f), torch.empty_like(m)))
part_inject = _op("part_inject", _part_inject,
                  lambda f, m: m.new_empty(*m.shape[:-1], f.shape[-1] + m.shape[-1]),
                  lambda ctx, g: part_inject_grad(g, *ctx.saved_tensors),
                  lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1]))


def _part_gather(feat: Tensor, labels: Tensor) -> Tensor:
    feat = _f32(feat, "feature_vectors")
    labels = labels.to(torch.int64).contiguous()
    B, K, F = feat.shape
    P = labels.numel() // B if B else 0
    out = torch.empty(*labels.shape, F, dtype=torch.float32, device=feat.device)
    C.call("ups_part_gather_fwd", feat.data_ptr(), labels.data_ptr(), out.data_ptr(), B, P, K, F, _stream(feat))
    return out


def _part_gather_setup(ctx, inputs, output):
    feat, labels = inputs
    ctx.save_for_backward(labels)
    ctx.K = feat.shape[1]


def _part_gather_bwd(ctx, g):
    """tf.gather is differentiable in `feature_vectors` (cub/code/nn.py:2469-2487): dfeat[b,k,:] is the sum of g over
    the pixels labelled k = the dense pooling of g with the one-hot mask (deterministic fixed-order sums)."""
    (labels,) = ctx.saved_tensors
    return part_pool(g.contiguous(), one_hot(labels, ctx.K), False, 1.0), None


part_gather = _op("part_gather", _part_gather, lambda f, l: f.new_empty(*l.shape, f.shape[-1]),
                  _part_gather_bwd, _part_gather_setup)


# ------------------------------------------------------------------ mask statistics (SURVEY.md 8f N1/N2)
def _mask_moments(probs: Tensor, scaling: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    probs, scaling = _f32(probs, "probs"), _f32(scaling, "scaling_factor")
    B, H, W, K = probs.shape
    mu = torch.empty(B, K, 2, dtype=torch.float32, device=probs.device)
    sigma = torch.empty(B, K, 2, 2, dtype=torch.float32, device=probs.device)
    moments = torch.empty(B, K, 5, dtype=torch.float32, device=probs.device)
    ws = _ws(C.workspace_bytes(C.OP_MOMENTS, B, H * W, K, 0), probs)
    C.call("ups_mask_moments_fwd", probs.data_ptr(), scaling.data_ptr(), mu.data_ptr(), sigma.data_ptr(),
           moments.data_ptr(), B, H, W, K, ws.data_ptr(), ws.numel(), _stream(probs))
    return mu, sigma, moments


def _mask_moments_fake(probs, scaling):
    B, H, W, K = probs.shape
    return probs.new_empty(B, K, 2), probs.new_empty(B, K, 2, 2), probs.new_empty(B, K, 5)


def _mask_moments_grad(g_mu: Tensor, g_sigma: Tensor, scaling: Tensor, moments: Tensor, shape: list[int]) -> Tensor:
    g_mu, g_sigma, scaling, moments = _f32(g_mu), _f32(g_sigma), _f32(scaling), _f32(moments)
    B, H, W, K = shape
    dprobs = torch.empty(B, H, W, K, dtype=torch.float32, device=moments.device)
    C.call("ups_mask_moments_bwd", g_mu.data_ptr(), g_sigma.data_ptr(), scaling.data_ptr(), moments.data_ptr(),
           dprobs.data_ptr(), B, H, W, K, _stream(g_mu))
    return dprobs


mask_moments_grad = _op("mask_moments_grad", _mask_moments_grad,
                        lambda gm, gs, s, m, shape: m.new_empty(shape))


def _mask_moments_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[1], output[2])
    ctx.shape = list(inputs[0].shape)


def _mask_moments_bwd(ctx, g_mu, g_sigma, g_moments):
    scaling, moments = ctx.saved_tensors
    g_mu = torch.zeros(moments.shape[0], moments.shape[1], 2, device=moments.device) if g_mu is None else g_mu
    g_sigma = torch.zeros(moments.shape[0], moments.shape[1], 2, 2, device=moments.device) if g_sigma is None else g_sigma
    return mask_moments_grad(g_mu, g_sigma, scaling, moments, ctx.shape), None


mask_moments = _op("mask_moments", _mask_moments, _mask_moments_fake, _mask_moments_bwd, _mask_moments_setup)


def _categorical_kl(probs: Tensor) -> Tensor:
    probs = _f32(probs, "probs")
    K = probs.shape[-1]
    n_pix = probs.numel() // K
    out = torch.empty((), dtype=torch.float32, device=probs.device)
    ws = _ws(C.workspace_bytes(C.OP_KL, 0, 0, K, 0), probs)
    C.call("ups_categorical_kl_fwd", probs.data_ptr(), out.data_ptr(), n_pix, K, ws.data_ptr(), ws.numel(), _stream(probs))
    return out


def _categorical_kl_grad(probs: Tensor, g: Tensor) -> Tensor:
    probs, g = _f32(probs), _f32(g)
    K = probs.shape[-1]
    d = torch.empty_like(probs)
    C.call("ups_categorical_kl_bwd", probs.data_ptr(), g.data_ptr(), d.data_ptr(), probs.numel() // K, K, _stream(probs))
    return d


categorical_kl_grad = _op("categorical_kl_grad", _categorical_kl_grad, lambda p, g: torch.empty_like(p))
categorical_kl = _op("categorical_kl", _categorical_kl, lambda p: p.new_empty(()),
                     lambda ctx, g: categorical_kl_grad(ctx.saved_tensors[0], g),
                     lambda ctx, inputs, output: ctx.save_for_backward(inputs[0]))


# ------------------------------------------------------------------ mask priors / sampling (SURVEY.md 8f N2/N3)
def _mumford_shah(x: Tensor, alpha: float, lambda_: float) -> Tuple[Tensor, Tensor, Tensor]:
    x = _f32(x, "x")
    B, H, W, K = x.shape
    r, s, c = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
    C.call("ups_mumford_shah_fwd", x.data_ptr(), alpha, lambda_, r.data_ptr(), s.data_ptr(), c.data_ptr(), None, None,
           B, H, W, K, None, 0, _stream(x))
    return r, s, c


def _mumford_shah_grad(x: Tensor, alpha: float, lambda_: float, g_r: Optional[Tensor], g_s: Optional[Tensor],
                       g_c: Optional[Tensor], g_sums: Optional[Tensor]) -> Tensor:
    x = _f32(x, "x")
    B, H, W, K = x.shape
    gs = [None if g is None else _f32(g) for g in (g_r, g_s, g_c, g_sums)]
    dx = torch.empty_like(x)
    C.call("ups_mumford_shah_bwd", x.data_ptr(), alpha, lambda_, *[_ptr(g) for g in gs], dx.data_ptr(), B, H, W, K,
           _stream(x))
    return dx


mumford_shah_grad = _op("mumford_shah_grad", _mumford_shah_grad, lambda x, a, l, gr, gs, gc, gq: torch.empty_like(x))


def _ms_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])
    ctx.alpha, ctx.lam = inputs[1], inputs[2]


mumford_shah = _op("mumford_shah", _mumford_shah,
                   lambda x, a, l: (torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)),
                   lambda ctx, g_r, g_s, g_c: (mumford_shah_grad(ctx.saved_tensors[0], ctx.alpha, ctx.lam, g_r, g_s, g_c,
                                                                 None), None, None),
                   _ms_setup)


def _mumford_shah_sums(x: Tensor, alpha: float, lambda_: float) -> Tensor:
    x = _f32(x, "x")
    B, H, W, K = x.shape
    sums = torch.empty(B, 4, K, dtype=torch.float32, device=x.device)
    ws = _ws(C.workspace_bytes(C.OP_MUMFORD_SHAH, B, H * W, K, 0), x)
    C.call("ups_mumford_shah_fwd", x.data_ptr(), alpha, lambda_, None, None, None, None, sums.data_ptr(), B, H, W, K,
           ws.data_ptr(), ws.numel(), _stream(x))
    return sums


mumford_shah_sums = _op("mumford_shah_sums", _mumford_shah_sums,
                        lambda x, a, l: x.new_empty(x.shape[0], 4, x.shape[3]),
                        lambda ctx, g: (mumford_shah_grad(ctx.saved_tensors[0], ctx.alpha, ctx.lam, None, None, None, g),
                                        None, None),
                        _ms_setup)


def _edge_set(x: Tensor, alpha: float, lambda_: float) -> Tensor:
    x = _f32(x, "x")
    B, H, W, K = x.shape
    e = torch.empty_like(x)
    C.call("ups_mumford_shah_fwd", x.data_ptr(), alpha, lambda_, None, None, None, e.data_ptr(), None, B, H, W, K,
           None, 0, _stream(x))
    return e


edge_set = _op("edge_set", _edge_set, lambda x, a, l: torch.empty_like(x))


def _logit_priors(mean: Tensor) -> Tensor:
    mean = _f32(mean, "mean")
    B, H, W, K = mean.shape
    out = torch.empty(3, dtype=torch.float32, device=mean.device)
    ws = _ws(C.workspace_bytes(C.OP_LOGIT_PRIORS, B, H * W, K, 0), mean)
    C.call("ups_logit_priors_fwd", mean.data_ptr(), out.data_ptr(), B, H, W, K, ws.data_ptr(), ws.numel(), _stream(mean))
    return out


def _logit_priors_grad(mean: Tensor, g: Tensor) -> Tensor:
    mean, g = _f32(mean), _f32(g)
    B, H, W, K = mean.shape
    d = torch.empty_like(mean)
    C.call("ups_logit_priors_bwd", mean.data_ptr(), g.data_ptr(), d.data_ptr(), B, H, W, K, _stream(mean))
    return d


logit_priors_grad = _op("logit_priors_grad", _logit_priors_grad, lambda m, g: torch.empty_like(m))
logit_priors = _op("logit_priors", _logit_priors, lambda m: m.new_empty(3),
                   lambda ctx, g: logit_priors_grad(ctx.saved_tensors[0], g),
                   lambda ctx, inputs, output: ctx.save_for_backward(inputs[0]))


def _mean_field_sample(mean: Tensor, eps: Tensor, noise_level: float) -> Tensor:
    mean, eps = _f32(mean, "mean"), _f32(eps, "eps")
    assert mean.shape == eps.shape, (list(mean.shape), list(eps.shape))
    out = torch.empty_like(mean)
    C.call("ups_mean_field_sample_fwd", mean.data_ptr(), eps.data_ptr(), noise_level, out.data_ptr(), mean.numel(),
           _stream(mean))
    return out


mean_field_sample = _op("mean_field_sample", _mean_field_sample, lambda m, e, n: torch.empty_like(m),
                        lambda ctx, g: (g, None, None), lambda ctx, inputs, output: None)


def _part_softmax_sampled(mean: Tensor, eps: Tensor, noise_level: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    mean, eps = _f32(mean, "mean"), _f32(eps, "eps")
    assert mean.shape == eps.shape, (list(mean.shape), list(eps.shape))
    K = mean.shape[-1]
    logits, probs, hard = torch.empty_like(mean), torch.empty_like(mean), torch.empty_like(mean)
    labels = torch.empty(mean.shape[:-1], dtype=torch.int64, device=mean.device)
    C.call("ups_part_softmax_sampled_fwd", mean.data_ptr(), eps.data_ptr(), noise_level, logits.data_ptr(),
           probs.data_ptr(), labels.data_ptr(), hard.data_ptr(), mean.numel() // K, K, _stream(mean))
    return logits, probs, labels, hard


def _pss_bwd(ctx, g_logits, g_probs, g_labels, g_hard):
    (p,) = ctx.saved_tensors
    g = g_probs if g_hard is None else (g_hard if g_probs is None else g_probs + g_hard)
    d = None if g is None else part_softmax_grad(p, g)
    if g_logits is not None:
        d = g_logits if d is None else d + g_logits
    return d, None, None


part_softmax_sampled = _op(
    "part_softmax_sampled", _part_softmax_sampled,
    lambda m, e, n: (torch.empty_like(m), torch.empty_like(m), m.new_empty(m.shape[:-1], dtype=torch.int64),
                     torch.empty_like(m)),
    _pss_bwd, lambda ctx, inputs, output: ctx.save_for_backward(output[1]))


# ------------------------------------------------------------------ the logit noise drawn on the device
# The draw is a pure function of (seed, draw, global pixel, part) (csrc/canon_math.cuh): ups_normal_philox_fwd writes it,
# ups_part_softmax_sampled_philox_fwd and the step's `_noise` kernels generate the same values in registers.  Seeds are
# unsigned 64-bit; the op schemas carry them as the int64 with the same bits.
def _seed_i64(seed: int) -> int:
    seed = int(seed)
    if not 0 <= seed < 2 ** 64:
        raise ValueError(f"seed must be in [0, 2**64), got {seed}")
    return seed - 2 ** 64 if seed >= 2 ** 63 else seed


def _normal_philox(seed: int, draw: int, pix_offset: int, n_pix: int, K: int, device: torch.device) -> Tensor:
    out = torch.empty(n_pix, K, dtype=torch.float32, device=device)
    if not out.is_cuda:
        raise C.UpsError("ups_b200: normal_philox needs a CUDA device (no CPU fallback exists)")
    C.call("ups_normal_philox_fwd", seed % 2 ** 64, draw, pix_offset, n_pix, K, out.data_ptr(), _stream(out))
    return out


normal_philox = _op("normal_philox", _normal_philox,
                    lambda seed, draw, off, n, K, device: torch.empty(n, K, dtype=torch.float32, device=device))


def _part_softmax_sampled_philox(mean: Tensor, seed: int, draw: int, pix_offset: int,
                                 noise_level: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    mean = _f32(mean, "mean")
    K = mean.shape[-1]
    logits, probs, hard = torch.empty_like(mean), torch.empty_like(mean), torch.empty_like(mean)
    labels = torch.empty(mean.shape[:-1], dtype=torch.int64, device=mean.device)
    C.call("ups_part_softmax_sampled_philox_fwd", mean.data_ptr(), seed % 2 ** 64, draw, pix_offset, noise_level,
           logits.data_ptr(), probs.data_ptr(), labels.data_ptr(), hard.data_ptr(), mean.numel() // K, K, _stream(mean))
    return logits, probs, labels, hard


def _pssp_bwd(ctx, g_logits, g_probs, g_labels, g_hard):
    return _pss_bwd(ctx, g_logits, g_probs, g_labels, g_hard)[0], None, None, None, None


part_softmax_sampled_philox = _op(
    "part_softmax_sampled_philox", _part_softmax_sampled_philox,
    lambda m, s, d, o, n: (torch.empty_like(m), torch.empty_like(m), m.new_empty(m.shape[:-1], dtype=torch.int64),
                           torch.empty_like(m)),
    _pssp_bwd, lambda ctx, inputs, output: ctx.save_for_backward(output[1]))


def _weak_xent(logits: Tensor, mode: int) -> Tensor:
    x = _f32(logits, "logits")
    K = x.shape[-1]
    n_pix = x.numel() // K
    out = torch.empty((), dtype=torch.float32, device=x.device)
    ws = _ws(C.workspace_bytes(C.OP_WEAK_XENT, 1, n_pix, K, 0), x)
    C.call("ups_weak_xent_fwd", x.data_ptr(), mode, out.data_ptr(), n_pix, K, ws.data_ptr(), ws.numel(), _stream(x))
    return out


def _weak_xent_grad(logits: Tensor, mode: int, g: Tensor) -> Tensor:
    x, g = _f32(logits), _f32(g)
    K = x.shape[-1]
    d = torch.empty_like(x)
    C.call("ups_weak_xent_bwd", x.data_ptr(), mode, g.data_ptr(), d.data_ptr(), x.numel() // K, K, _stream(x))
    return d


def _wx_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])
    ctx.mode = inputs[1]


weak_xent_grad = _op("weak_xent_grad", _weak_xent_grad, lambda x, m, g: torch.empty_like(x))
weak_xent = _op("weak_xent", _weak_xent, lambda x, m: x.new_empty(()),
                lambda ctx, g: (weak_xent_grad(ctx.saved_tensors[0], ctx.mode, g), None), _wx_setup)


def _mask2rgb(mask: Tensor, table: Tensor, make_hot: bool) -> Tensor:
    mask, table = _f32(mask, "mask"), _f32(table, "colors")
    K = mask.shape[-1]
    assert list(table.shape) == [K, 3], list(table.shape)
    out = torch.empty(*mask.shape[:-1], 3, dtype=torch.float32, device=mask.device)
    C.call("ups_mask2rgb_fwd", mask.data_ptr(), table.data_ptr(), int(make_hot), out.data_ptr(), mask.numel() // K, K,
           _stream(mask))
    return out


mask2rgb = _op("mask2rgb", _mask2rgb, lambda m, t, h: m.new_empty(*m.shape[:-1], 3))


# ------------------------------------------------------------------ decoder first conv on the part assignment (N4)
def _inject_conv_table(feat: Tensor, V: Tensor) -> Tensor:
    feat, V = _f32(feat, "feature_vectors"), _f32(V, "V")
    B, K, F = feat.shape
    Co = V.shape[-1]
    G = torch.empty(B, 9, K, Co, dtype=torch.float32, device=feat.device)
    C.call("ups_inject_conv_table_fwd", feat.data_ptr(), V.data_ptr(), G.data_ptr(), B, K, F, Co, _stream(feat))
    return G


def _inject_conv_table_grad(dG: Tensor, feat: Tensor, V: Tensor) -> Tuple[Tensor, Tensor]:
    dG, feat, V = _f32(dG), _f32(feat), _f32(V)
    B, K, F = feat.shape
    Co = V.shape[-1]
    dfeat, dV = torch.empty_like(feat), torch.empty_like(V)
    C.call("ups_inject_conv_table_bwd", dG.data_ptr(), feat.data_ptr(), V.data_ptr(), dfeat.data_ptr(), dV.data_ptr(),
           B, K, F, Co, _stream(dG))
    return dfeat, dV


inject_conv_table_grad = _op("inject_conv_table_grad", _inject_conv_table_grad,
                             lambda g, f, v: (torch.empty_like(f), torch.empty_like(v)))
inject_conv_table = _op("inject_conv_table", _inject_conv_table,
                        lambda f, v: f.new_empty(f.shape[0], 9, f.shape[1], v.shape[-1]),
                        lambda ctx, g: inject_conv_table_grad(g, *ctx.saved_tensors),
                        lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1]))


def _inject_conv_apply(mask: Tensor, G: Tensor, bias: Tensor) -> Tensor:
    mask, G, bias = _f32(mask, "mask"), _f32(G, "G"), _f32(bias, "b")
    B, H, W, K = mask.shape
    Co = G.shape[-1]
    out = torch.empty(B, H, W, Co, dtype=torch.float32, device=mask.device)
    C.call("ups_inject_conv_fwd", mask.data_ptr(), G.data_ptr(), bias.data_ptr(), out.data_ptr(), B, H, W, K, Co,
           _stream(mask))
    return out


def _inject_conv_apply_grad(g_out: Tensor, mask: Tensor, G: Tensor, probs: Optional[Tensor],
                            g_extra: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor]:
    g_out, mask, G = _f32(g_out), _f32(mask), _f32(G)
    probs = None if probs is None else _f32(probs)
    g_extra = None if g_extra is None else _f32(g_extra)
    B, H, W, K = mask.shape
    Co = G.shape[-1]
    dmask, dG = torch.empty_like(mask), torch.empty_like(G)
    db = torch.empty(Co, dtype=torch.float32, device=mask.device)
    ws = _ws(C.inject_conv_workspace_bytes(B, H, W, K, Co), mask)
    C.call("ups_inject_conv_bwd", g_out.data_ptr(), mask.data_ptr(), G.data_ptr(), _ptr(probs), _ptr(g_extra),
           dmask.data_ptr(), dG.data_ptr(), db.data_ptr(), B, H, W, K, Co, ws.data_ptr(), ws.numel(), _stream(g_out))
    return dmask, dG, db


inject_conv_apply_grad = _op(
    "inject_conv_apply_grad", _inject_conv_apply_grad,
    lambda g, m, G, p, e: (torch.empty_like(m), torch.empty_like(G), G.new_empty(G.shape[-1])))
inject_conv_apply = _op("inject_conv_apply", _inject_conv_apply,
                        lambda m, G, b: m.new_empty(*m.shape[:-1], G.shape[-1]),
                        lambda ctx, g: inject_conv_apply_grad(g, *ctx.saved_tensors, None, None),
                        lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1]))


def _decode_conv(logits: Tensor, G: Tensor, bias: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """softmax -> labels -> ST(hard_max) -> first decoder conv, the decode side of the step with the conv folded in."""
    probs, labels, hard = _part_softmax_full(logits)
    return probs, labels, hard, _inject_conv_apply(hard, G, bias)


def _decode_conv_bwd(ctx, g_probs, g_labels, g_hard, g_out):
    probs, hard, G = ctx.saved_tensors
    g_extra = g_probs if g_hard is None else (g_hard if g_probs is None else g_probs + g_hard)
    if g_out is None:
        return (None if g_extra is None else part_softmax_grad(probs, g_extra)), None, None
    dlogits, dG, db = inject_conv_apply_grad(g_out, hard, G, probs, g_extra)
    return dlogits, dG, db


decode_conv = _op(
    "decode_conv", _decode_conv,
    lambda x, G, b: (torch.empty_like(x), x.new_empty(x.shape[:-1], dtype=torch.int64), torch.empty_like(x),
                     x.new_empty(*x.shape[:-1], G.shape[-1])),
    _decode_conv_bwd, lambda ctx, inputs, output: ctx.save_for_backward(output[0], output[2], inputs[1]))


# ------------------------------------------------------------------ encoder first conv on the masked part images (N4)
def _parts_conv(image: Tensor, mask: Tensor, V: Tensor, bias: Tensor) -> Tensor:
    image, mask, V, bias = _f32(image, "image"), _f32(mask, "mask"), _f32(V, "V"), _f32(bias, "b")
    B, H, W, K = mask.shape
    Cin, Co = image.shape[-1], V.shape[-1]
    out = torch.empty(K * B, H, W, Co, dtype=torch.float32, device=image.device)
    C.call("ups_parts_conv_fwd", image.data_ptr(), mask.data_ptr(), V.data_ptr(), bias.data_ptr(), out.data_ptr(),
           B, H, W, K, Cin, Co, _stream(image))
    return out


def _parts_conv_grad(g_out: Tensor, image: Tensor, mask: Tensor, V: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    g_out, image, mask, V = _f32(g_out), _f32(image), _f32(mask), _f32(V)
    B, H, W, K = mask.shape
    Cin, Co = image.shape[-1], V.shape[-1]
    dmask, dV = torch.empty_like(mask), torch.empty_like(V)
    db = torch.empty(Co, dtype=torch.float32, device=mask.device)
    ws = _ws(C.parts_conv_bwd_workspace_bytes(B, H, W, K, Co), mask)
    C.call("ups_parts_conv_bwd", g_out.data_ptr(), image.data_ptr(), mask.data_ptr(), V.data_ptr(), None, None,
           dmask.data_ptr(), dV.data_ptr(), db.data_ptr(), B, H, W, K, Cin, Co, ws.data_ptr(), ws.numel(), _stream(g_out))
    return dmask, dV, db


parts_conv_grad = _op("parts_conv_grad", _parts_conv_grad,
                      lambda g, i, m, v: (torch.empty_like(m), torch.empty_like(v), v.new_empty(v.shape[-1])))


def _parts_conv_bwd(ctx, g):
    if ctx.needs_input_grad[0]:
        raise C.UpsError("ups::parts_conv: no gradient with respect to the image (the reference's inputs are placeholders)")
    dmask, dV, db = parts_conv_grad(g, *ctx.saved_tensors)
    return None, dmask, dV, db


parts_conv = _op("parts_conv", _parts_conv,
                 lambda i, m, v, b: i.new_empty(m.shape[-1] * m.shape[0], m.shape[1], m.shape[2], v.shape[-1]),
                 _parts_conv_bwd, lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1], inputs[2]))


# ------------------------------------------------------------------ patch masks (SURVEY.md 8f N1: draw_rect)
def _draw_rect(centers: Tensor, ph: int, pw: int, H: int, W: int) -> Tensor:
    if not centers.is_cuda:
        raise C.UpsError("ups_b200: centers must be a CUDA tensor (no CPU fallback exists)")
    centers = centers.to(torch.int32).contiguous()
    N = centers.shape[0]
    out = torch.empty(N, H, W, dtype=torch.float32, device=centers.device)
    C.call("ups_draw_rect_fwd", centers.data_ptr(), out.data_ptr(), N, int(ph), int(pw), int(H), int(W), _stream(centers))
    return out


draw_rect = _op("draw_rect", _draw_rect, lambda c, ph, pw, H, W: c.new_empty(c.shape[0], H, W, dtype=torch.float32))


# ------------------------------------------------------------------ the step's two sides in the reference model's order
# model.py:426-485 runs the appearance encoder between the sides: part_encode (K2: m1, the part images and their mean pool)
# feeds e_alpha, whose output feeds part_decode (K3: m0, labels0 and the injected map).  Each side is one op with autograd
# (K5 / K4 as its backward) on the kernels step.kernel_route picks, the rule PartStep follows, so both produce the same
# bits.  Outputs and workspaces come from the caching allocator on every call: two forwards may precede their backwards.
# A padded part count (e.g. 25 on the kernels of 32) returns views [..., :K] of row-pitched buffers, as PartStep does.
#
# Noise (the sampled logits of MeanFieldDistribution.sample, model.py:420-421): `noise` = NOISE_NONE, NOISE_INT (the
# seed is `seed_value`, passed by value) or NOISE_DEVICE (the seed is the one int64 element of `seed`, read by the kernels
# from device memory, so a captured CUDA graph draws with whatever that tensor holds at replay).  Decode draws 0, encode
# draws 1: the draws of PartStep.forward(noise_seed=...).
NOISE_NONE, NOISE_INT, NOISE_DEVICE = 0, 1, 2


def _noise_call(name, noise, seed, seed_value, *args):
    """Call entry point `name` noise-free, or its `_noise` / `_noise_dseed` form: the same arguments with
    (seed, sample_offset, noise_level) inserted before the stream (`args` ends with those three and the stream)."""
    *head, offset, level, st = args
    if noise == NOISE_NONE:
        C.call(name, *head, st)
    elif noise == NOISE_INT:
        C.call(name[:-len("_rows")] + "_noise", *head, seed_value % 2 ** 64, offset, level, st)
    else:
        C.call(name[:-len("_rows")] + "_noise_dseed", *head, seed.data_ptr(), offset, level, st)


def _softmax_noise(logits, noise, seed, seed_value, draw, pix_offset, level, probs, labels, hard, n_pix, K, st):
    """The generic kernels' softmax of the logits, or of the sampled logits (the step's draw `draw`)."""
    if noise == NOISE_NONE:
        C.call("ups_part_softmax_fwd", logits.data_ptr(), probs.data_ptr(), _ptr(labels), _ptr(hard), n_pix, K, st)
    elif noise == NOISE_INT:
        C.call("ups_part_softmax_sampled_philox_fwd", logits.data_ptr(), seed_value % 2 ** 64, draw, pix_offset, level,
               None, probs.data_ptr(), _ptr(labels), _ptr(hard), n_pix, K, st)
    else:
        C.call("ups_part_softmax_sampled_philox_fwd_dseed", logits.data_ptr(), seed.data_ptr(), draw, pix_offset, level,
               None, probs.data_ptr(), _ptr(labels), _ptr(hard), n_pix, K, st)


def _check_noise(noise: int, seed: Optional[Tensor], device):
    if noise == NOISE_INT and torch.cuda.is_current_stream_capturing():
        raise C.UpsError("ups_b200: an int noise_seed is frozen into a captured CUDA graph (every replay would draw the "
                         "same noise); pass the seed as a one-element int64 CUDA tensor")
    if noise == NOISE_DEVICE:
        if seed is None or seed.dtype != torch.int64 or seed.numel() != 1 or seed.device != device:
            raise C.UpsError("ups_b200: a device noise_seed is a one-element int64 tensor on the logits' device")
        if not seed.is_contiguous():
            raise C.UpsError("ups_b200: the device noise_seed must be contiguous")


def _pitched(t: Tensor, Kp: int, st) -> Tensor:
    """A [.., K] tensor as the base of a row-pitched [.., Kp] buffer: itself when it already is a view [..., :K] of
    such a buffer (what the padded forwards return), else a zero-padded copy."""
    K = t.shape[-1]
    rows = t.numel() // K if K else 0
    if (t.stride(-1) == 1 and all(t.stride(i) == Kp * math.prod(t.shape[i + 1:-1]) for i in range(t.dim() - 1))
            and t.untyped_storage().nbytes() >= (t.storage_offset() + rows * Kp) * t.element_size()):
        return t
    t = t.contiguous()
    out = torch.empty(*t.shape[:-1], Kp, dtype=t.dtype, device=t.device)
    C.call("ups_copy_rows", t.data_ptr(), K, out.data_ptr(), Kp, t.numel() // K if K else 0, K, Kp - K, 0.0, st)
    return out


def _pad_rows(t: Tensor, n: int, pitch: int, st) -> Tensor:
    """Contiguous [.., n] -> [.., pitch], the columns n.. zero."""
    t = t.contiguous()
    out = torch.empty(*t.shape[:-1], pitch, dtype=t.dtype, device=t.device)
    C.call("ups_copy_rows", t.data_ptr(), n, out.data_ptr(), pitch, t.numel() // n, n, pitch - n, 0.0, st)
    return out


def _hard_of(probs: Tensor, st) -> Tensor:
    """ST(hard_max(probs)), bit for bit what the softmax kernels write as `hard`."""
    K = probs.shape[-1]
    h = torch.empty_like(probs)
    C.call("ups_hard_max_fwd", probs.data_ptr(), h.data_ptr(), probs.numel() // K, K, st)
    C.call("ups_straight_through_fwd", h.data_ptr(), probs.data_ptr(), h.data_ptr(), h.numel(), st)
    return h


def _padded_fake(shape, K, Kp, like):
    """Fake of a view [..., :n] of a [..., n + Kp - K] buffer (n = shape[-1])."""
    n = shape[-1]
    return like.new_empty(*shape[:-1], n + Kp - K)[..., :n]


# ---- encode side: K2 forward, K5 backward
def _part_encode(l1: Tensor, image1: Tensor, noise: int, seed: Optional[Tensor], seed_value: int, noise_level: float,
                 sample_offset: int) -> Tuple[Tensor, Tensor, Tensor]:
    l1, img = _f32(l1, "logits1"), _f32(image1, "image1")
    _check_noise(noise, seed, l1.device)
    B, H, W, K = l1.shape
    P = H * W
    st = _stream(l1)
    route, Kk = kernel_route(K, None, P)
    dev = dict(dtype=torch.float32, device=l1.device)
    parts = torch.empty(K * B, H, W, 3, **dev)
    if route == "generic":
        m1, hard = torch.empty_like(l1), torch.empty_like(l1)
        pooled = torch.empty(B, K, 3, **dev)
        _softmax_noise(l1, noise, seed, seed_value, 1, sample_offset * P, noise_level, m1, None, hard, B * P, K, st)
        C.call("ups_mask_parts_fwd", img.data_ptr(), hard.data_ptr(), parts.data_ptr(), B, P, K, 3, 1, st)
        ws = _ws(C.workspace_bytes(C.OP_POOL, B, P, K, 3), l1)
        C.call("ups_part_pool_fwd", img.data_ptr(), hard.data_ptr(), pooled.data_ptr(), B, P, K, 3, 0, 1.0 / P,
               ws.data_ptr(), ws.numel(), st)
        return m1, parts, pooled
    m1 = torch.empty(B, H, W, Kk, **dev)
    pooled = torch.empty(B, Kk, 3, **dev)
    ws = _ws(C.workspace_bytes(C.OP_STEP, B, P, Kk, 3), l1)
    _noise_call("ups_step_encode_fwd_rows", noise, seed, seed_value, l1.data_ptr(), K, img.data_ptr(), m1.data_ptr(),
                parts.data_ptr(), pooled.data_ptr(), B, P, Kk, K, ws.data_ptr(), ws.numel(), sample_offset, noise_level, st)
    return m1[..., :K], parts, pooled[:, :K]


def _part_encode_fake(l1, image1, noise, seed, seed_value, noise_level, sample_offset):
    B, H, W, K = l1.shape
    route, Kk = kernel_route(K, None, H * W)
    return (_padded_fake(l1.shape, K, Kk, l1), l1.new_empty(K * B, H, W, 3), l1.new_empty(B, Kk, 3)[:, :K])


def _part_encode_grad(g_parts: Tensor, g_pooled: Optional[Tensor], g_m1: Optional[Tensor], m1: Tensor, image1: Tensor,
                      want_dimg: bool) -> Tuple[Tensor, Tensor]:
    g_parts, img = _f32(g_parts, "g_parts"), _f32(image1, "image1")
    g_pooled = None if g_pooled is None else _f32(g_pooled, "g_pooled")
    g_m1 = None if g_m1 is None else _f32(g_m1, "g_m1")
    B, H, W, K = m1.shape
    P = H * W
    st = _stream(img)
    route, Kk = kernel_route(K, None, P)
    dimg = torch.empty(B, H, W, 3, dtype=torch.float32, device=img.device) if want_dimg else img.new_empty(0)
    if route == "generic":
        m1 = _f32(m1, "m1")
        hard = _hard_of(m1, st)
        dm, dl1 = torch.empty_like(m1), torch.empty_like(m1)
        C.call("ups_mask_parts_bwd", g_parts.data_ptr(), img.data_ptr(), hard.data_ptr(), _ptr(dimg) if want_dimg else None,
               dm.data_ptr(), B, P, K, 3, 1, st)
        dm2 = None
        if g_pooled is not None:
            dm2 = torch.empty_like(m1)
            dfm = torch.empty_like(dimg) if want_dimg else None
            C.call("ups_part_pool_bwd", g_pooled.data_ptr(), img.data_ptr(), hard.data_ptr(), _ptr(dfm), dm2.data_ptr(),
                   B, P, K, 3, 0, 1.0 / P, st)
            if want_dimg:
                C.call("ups_axpy", dfm.data_ptr(), dimg.data_ptr(), dimg.numel(), 1.0, st)
        C.call("ups_part_softmax_bwd2", m1.data_ptr(), dm.data_ptr(), _ptr(dm2), _ptr(g_m1), dl1.data_ptr(), B * P, K, st)
        return dl1, dimg
    m1p = _pitched(m1, Kk, st)
    if g_pooled is not None and Kk != K:
        g_pooled = _pad_rows(g_pooled.reshape(B, K * 3), K * 3, Kk * 3, st)
    dl1 = torch.empty(B, H, W, Kk, dtype=torch.float32, device=img.device)
    C.call("ups_step_encode_bwd_rows", g_parts.data_ptr(), _ptr(g_pooled), img.data_ptr(), m1p.data_ptr(), _ptr(g_m1), K,
           dl1.data_ptr(), _ptr(dimg) if want_dimg else None, B, P, Kk, K, st)
    return dl1[..., :K], dimg


def _part_encode_grad_fake(g_parts, g_pooled, g_m1, m1, image1, want_dimg):
    B, H, W, K = m1.shape
    route, Kk = kernel_route(K, None, H * W)
    return _padded_fake(m1.shape, K, Kk, m1), (m1.new_empty(B, H, W, 3) if want_dimg else m1.new_empty(0))


part_encode_grad = _op("part_encode_grad", _part_encode_grad, _part_encode_grad_fake)


def _part_encode_setup(ctx, inputs, output):
    l1, image1 = inputs[0], inputs[1]
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(output[0], image1)
    ctx.parts_shape = tuple(output[1].shape)


def _part_encode_bwd(ctx, g_m1, g_parts, g_pooled):
    m1, image1 = ctx.saved_tensors
    want_dimg = ctx.needs_input_grad[1]
    if g_m1 is None and g_parts is None and g_pooled is None:
        return (None,) * 7
    if g_parts is None:
        g_parts = m1.new_zeros(ctx.parts_shape)
    dl1, dimg = part_encode_grad(g_parts, g_pooled, g_m1, m1, image1, want_dimg)
    return dl1, (dimg if want_dimg else None), None, None, None, None, None


part_encode = _op("part_encode", _part_encode, _part_encode_fake, _part_encode_bwd, _part_encode_setup)


# ---- decode side: K3 forward, K4 backward
def _part_decode(l0: Tensor, feat: Tensor, noise: int, seed: Optional[Tensor], seed_value: int, noise_level: float,
                 sample_offset: int) -> Tuple[Tensor, Tensor, Tensor]:
    l0, feat = _f32(l0, "logits0"), _f32(feat, "feature_vectors")
    _check_noise(noise, seed, l0.device)
    B, H, W, K = l0.shape
    F = feat.shape[-1]
    P = H * W
    st = _stream(l0)
    route, Kk = kernel_route(K, F, P)
    dev = dict(dtype=torch.float32, device=l0.device)
    labels = torch.empty(B, H, W, dtype=torch.int64, device=l0.device)
    if route == "generic":
        m0, hard = torch.empty_like(l0), torch.empty_like(l0)
        inj = torch.empty(B, H, W, F + K, **dev)
        _softmax_noise(l0, noise, seed, seed_value, 0, sample_offset * P, noise_level, m0, labels, hard, B * P, K, st)
        C.call("ups_part_inject_fwd", feat.data_ptr(), hard.data_ptr(), inj.data_ptr(), B, P, K, F, st)
        return m0, labels, inj
    if Kk != K:
        feat = _pad_rows(feat.reshape(B, K * F), K * F, Kk * F, st)
    m0 = torch.empty(B, H, W, Kk, **dev)
    inj = torch.empty(B, H, W, F + Kk, **dev)
    _noise_call("ups_step_decode_fwd_rows", noise, seed, seed_value, l0.data_ptr(), K, feat.data_ptr(), m0.data_ptr(),
                labels.data_ptr(), inj.data_ptr(), B, P, Kk, F, sample_offset, noise_level, st)
    return m0[..., :K], labels, inj[..., :F + K]


def _part_decode_fake(l0, feat, noise, seed, seed_value, noise_level, sample_offset):
    B, H, W, K = l0.shape
    F = feat.shape[-1]
    route, Kk = kernel_route(K, F, H * W)
    return (_padded_fake(l0.shape, K, Kk, l0), l0.new_empty(B, H, W, dtype=torch.int64),
            _padded_fake((B, H, W, F + K), K, Kk, l0))


def _part_decode_grad(g_inj: Tensor, g_m0: Optional[Tensor], m0: Tensor, feat: Tensor) -> Tuple[Tensor, Tensor]:
    g_inj, feat = _f32(g_inj, "g_inj"), _f32(feat, "feature_vectors")
    g_m0 = None if g_m0 is None else _f32(g_m0, "g_m0")
    B, H, W, K = m0.shape
    F = feat.shape[-1]
    P = H * W
    st = _stream(feat)
    route, Kk = kernel_route(K, F, P)
    if route == "generic":
        m0 = _f32(m0, "m0")
        hard = _hard_of(m0, st)
        dm, dl0, dfeat = torch.empty_like(m0), torch.empty_like(m0), torch.empty_like(feat)
        ws = _ws(C.workspace_bytes(C.OP_INJECT_BWD, B, P, K, F), feat)
        C.call("ups_part_inject_bwd", g_inj.data_ptr(), feat.data_ptr(), hard.data_ptr(), dfeat.data_ptr(), dm.data_ptr(),
               B, P, K, F, ws.data_ptr(), ws.numel(), st)
        C.call("ups_part_softmax_bwd2", m0.data_ptr(), dm.data_ptr(), _ptr(g_m0), None, dl0.data_ptr(), B * P, K, st)
        return dl0, dfeat
    m0p = _pitched(m0, Kk, st)
    if Kk != K:
        g_inj = _pad_rows(g_inj, F + K, F + Kk, st)
        feat = _pad_rows(feat.reshape(B, K * F), K * F, Kk * F, st)
    dl0 = torch.empty(B, H, W, Kk, dtype=torch.float32, device=feat.device)
    dfeat = torch.empty(B, Kk, F, dtype=torch.float32, device=feat.device)
    ws = _ws(C.workspace_bytes(C.OP_STEP, B, P, Kk, F), feat)
    C.call("ups_step_decode_bwd_tc_rows" if decode_bwd_tc_ok(Kk, F, P) else "ups_step_decode_bwd_rows",
           g_inj.data_ptr(), m0p.data_ptr(), _ptr(g_m0), K, feat.data_ptr(), dl0.data_ptr(), dfeat.data_ptr(),
           B, P, Kk, F, ws.data_ptr(), ws.numel(), st)
    return dl0[..., :K], dfeat[:, :K]


def _part_decode_grad_fake(g_inj, g_m0, m0, feat):
    B, H, W, K = m0.shape
    F = feat.shape[-1]
    route, Kk = kernel_route(K, F, H * W)
    return _padded_fake(m0.shape, K, Kk, m0), m0.new_empty(B, Kk, F)[:, :K]


part_decode_grad = _op("part_decode_grad", _part_decode_grad, _part_decode_grad_fake)


def _part_decode_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(output[0], inputs[1])
    ctx.inj_shape = tuple(output[2].shape)


def _part_decode_bwd(ctx, g_m0, g_labels, g_inj):
    m0, feat = ctx.saved_tensors
    if g_m0 is None and g_inj is None:
        return (None,) * 7
    if g_inj is None:
        g_inj = m0.new_zeros(ctx.inj_shape)
    dl0, dfeat = part_decode_grad(g_inj, g_m0, m0, feat)
    return dl0, dfeat, None, None, None, None, None


part_decode = _op("part_decode", _part_decode, _part_decode_fake, _part_decode_bwd, _part_decode_setup)
