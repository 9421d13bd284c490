"""The fused per-step part-disentanglement path (forward + backward) on one GPU.

What the reference builds per training step in TrainModel.define_graph
(cub/code/SB_model48i/model.py:337,426-485) and differentiates with tf.gradients:

    warped          = make_tps(views)                                   model.py:282-311
    m0, m1          = softmax(l0), softmax(l1)                          model.py:426-430
    labels0         = argmax(m0, 3)                                     model.py:447,470
    m0h, m1h        = ST(hard_max(m0)), ST(hard_max(m1))                model.py:434-436,453-455
    parts           = apply_partwise-fold(mask_parts(warped[1], m1h))   model.py:478 ; nn.py:100-103
    pooled          = mean_hw(parts)        (tail of e_alpha)           model.py:50-52
    inj             = concat(sum_k unpool_features(feat, m0h), m0h)     model.py:482-484
    [h0             = conv2d(inj, V) + b   (first layer of `dd`)        model.py:96,485 ; nn.py:617-664
                      with first_conv=Co: computed from m0h and feat directly, `inj` is never formed (SURVEY 8f N4)]

With a noise seed, l0 and l1 are the means of MeanFieldDistribution and the step samples them itself
(model.py:420-421, cub/code/nn.py:1421-1427): m0, m1 = softmax(l0 + noise_level*eps0), softmax(l1 + noise_level*eps1)
with eps drawn in registers from (seed, side, global pixel, part) (csrc/canon_math.cuh, ups_normal_philox_fwd).

The CNNs between those pieces are not part of the path: `l0`, `l1` (mask decoder output) and
`feat` (appearance encoder output) are inputs, and the cotangents of every output are inputs
to `backward`.  All buffers are allocated once in __init__ (180 GB HBM: the B=256 CUB step
holds ~3.6 GB); forward/backward only enqueue kernels on the current stream.
"""
import os

import torch

from . import _cabi as C


def kernel_route(K, F, P, first_conv=0, encoder_conv=0):
    """The kernels that run a step side of K parts (F feature channels, None for the encode side, which has none) on
    samples of P pixels: ("fused", K) for the fused kernels (K in {8,16,32}); ("padded", Kp) for a part count below 32
    that is not a power of two, run on the fused kernels of the next power of two Kp with -inf logits in the padding
    parts; ("generic", K) for everything else (the stand-alone softmax / mask_parts / pool / inject kernels).  The one
    rule that PartStep and the ups::part_encode / ups::part_decode ops both follow.  UPS_PAD_K=0 keeps padded part
    counts on the generic kernels."""
    f_ok = F is None or F in (16, 32, 64)
    if K in (8, 16, 32) and f_ok and P % 32 == 0:
        return "fused", K
    if (not first_conv and not encoder_conv and 1 <= K < 32 and f_ok and P % 32 == 0
            and os.environ.get("UPS_PAD_K", "1") != "0"):
        return "padded", 8 if K <= 8 else 16 if K <= 16 else 32
    return "generic", K


def decode_bwd_tc_ok(K, F, P):
    """Whether K4 (the decode side's backward on the fused kernels) can run as the persistent TMA + tcgen05/TMEM
    pipeline; otherwise it runs on the CUDA cores."""
    return K in (16, 32) and F == 64 and P % 128 == 0


# ------------------------------------------------------------------ the launch sequence of each step side
# Written once, called by PartStep with its persistent buffers and by the ups::part_* / ups::*_conv ops with fresh ones.
# A launcher allocates nothing: outputs, scratch and workspaces, and the padded copies of a padded part count, come from
# the caller.  `route` is kernel_route's: the fused kernels of K parts ("fused", "padded": logits and cotangents read in
# rows of `row` floats, `planes` part planes written) or the generic ones ("generic", through the hard mask `hard`).
# `noise` is None (the noise-free step) or (seed, sample_offset, noise_level): the logits are the means and the kernels
# add noise_level * eps, eps drawn from (seed, draw, global pixel (sample_offset + b) * P + p, part); decode draws 0,
# encode draws 1.  The seed is an int passed by value, or a one-element int64 CUDA tensor that the `_dseed` entry points
# read on the device (a captured CUDA graph then draws with whatever that tensor holds at replay).
def _ptr(t):
    return None if t is None else t.data_ptr()


def _seed_i64(seed):
    """An unsigned 64-bit seed as the int64 with the same bits (what the op schemas carry); out of range raises."""
    seed = int(seed)
    if not 0 <= seed < 2 ** 64:
        raise ValueError(f"seed must be in [0, 2**64), got {seed}")
    return seed - 2 ** 64 if seed >= 2 ** 63 else seed


def _seed_arg(seed):
    return seed.data_ptr() if isinstance(seed, torch.Tensor) else seed % 2 ** 64


def call_rows(name, noise, *args):
    """Call the `_rows` entry point `name`, or with noise its `_noise` / `_noise_dseed` form: the same kernel, reading the
    logits as means, with (seed, sample_offset, noise_level) inserted before the stream."""
    if noise is None:
        C.call(name, *args)
    else:
        seed, offset, level = noise
        suffix = "_noise_dseed" if isinstance(seed, torch.Tensor) else "_noise"
        C.call(name[:-len("_rows")] + suffix, *args[:-1], _seed_arg(seed), offset, level, args[-1])


def part_softmax_fwd(noise, draw, logits, probs, labels, hard, B, P, K, st):
    """The generic softmax of the logits (probs [, labels] [, hard = ST(hard_max)]), or of the sampled logits."""
    if noise is None:
        C.call("ups_part_softmax_fwd", logits.data_ptr(), probs.data_ptr(), _ptr(labels), _ptr(hard), B * P, K, st)
        return
    seed, offset, level = noise
    C.call("ups_part_softmax_sampled_philox_fwd_dseed" if isinstance(seed, torch.Tensor) else
           "ups_part_softmax_sampled_philox_fwd", logits.data_ptr(), _seed_arg(seed), draw, offset * P, level, None,
           probs.data_ptr(), _ptr(labels), _ptr(hard), B * P, K, st)


def encode_fwd(route, noise, l1, img1, m1, parts, pooled, hard, ws, B, P, K, row, planes, st):
    """K2 (m1, the part images, their mean pool), or softmax -> mask_parts -> part_pool."""
    if route != "generic":
        call_rows("ups_step_encode_fwd_rows", noise, l1.data_ptr(), row, img1.data_ptr(), m1.data_ptr(), parts.data_ptr(),
                  pooled.data_ptr(), B, P, K, planes, ws.data_ptr(), ws.numel(), st)
        return
    part_softmax_fwd(noise, 1, l1, m1, None, hard, B, P, K, st)
    C.call("ups_mask_parts_fwd", img1.data_ptr(), hard.data_ptr(), parts.data_ptr(), B, P, K, 3, 1, st)
    C.call("ups_part_pool_fwd", img1.data_ptr(), hard.data_ptr(), pooled.data_ptr(), B, P, K, 3, 0, 1.0 / P,
           ws.data_ptr(), ws.numel(), st)


def encode_bwd(route, g_parts, g_pooled, g_m1, img1, m1, hard, dl1, dimg1, dm, dm2, dfm, B, P, K, row, planes, st):
    """K5 (dl1 [, dimg1]), or mask_parts_bwd [+ part_pool_bwd into dm2 (its image cotangent dfm added to dimg1)] ->
    softmax_bwd2 of dm + dm2 + g_m1.  An undefined cotangent (None) or dimg1 = None reaches the kernels as a null pointer."""
    if route != "generic":
        C.call("ups_step_encode_bwd_rows", g_parts.data_ptr(), _ptr(g_pooled), img1.data_ptr(), m1.data_ptr(), _ptr(g_m1),
               row, dl1.data_ptr(), _ptr(dimg1), B, P, K, planes, st)
        return
    C.call("ups_mask_parts_bwd", g_parts.data_ptr(), img1.data_ptr(), hard.data_ptr(), _ptr(dimg1), dm.data_ptr(),
           B, P, K, 3, 1, st)
    if g_pooled is None:
        dm2 = None
    else:
        C.call("ups_part_pool_bwd", g_pooled.data_ptr(), img1.data_ptr(), hard.data_ptr(),
               _ptr(dfm if dimg1 is not None else None), dm2.data_ptr(), B, P, K, 3, 0, 1.0 / P, st)
        if dimg1 is not None:
            C.call("ups_axpy", dfm.data_ptr(), dimg1.data_ptr(), dimg1.numel(), 1.0, st)
    C.call("ups_part_softmax_bwd2", m1.data_ptr(), dm.data_ptr(), _ptr(dm2), _ptr(g_m1), dl1.data_ptr(), B * P, K, st)


def decode_fwd(route, noise, l0, feat, m0, labels0, inj, hard, B, P, K, F, row, st):
    """K3 (m0, labels0, the injected map), or softmax -> part_inject."""
    if route != "generic":
        call_rows("ups_step_decode_fwd_rows", noise, l0.data_ptr(), row, feat.data_ptr(), m0.data_ptr(), labels0.data_ptr(),
                  inj.data_ptr(), B, P, K, F, st)
        return
    part_softmax_fwd(noise, 0, l0, m0, labels0, hard, B, P, K, st)
    C.call("ups_part_inject_fwd", feat.data_ptr(), hard.data_ptr(), inj.data_ptr(), B, P, K, F, st)


def decode_bwd(route, tc, g_inj, g_m0, m0, hard, feat, dl0, dfeat, dm, ws, B, P, K, F, row, st):
    """K4 (dl0, dfeat) on tcgen05 (tc) or on the CUDA cores, or part_inject_bwd -> softmax_bwd2 of dm + g_m0."""
    if route != "generic":
        C.call("ups_step_decode_bwd_tc_rows" if tc else "ups_step_decode_bwd_rows", g_inj.data_ptr(), m0.data_ptr(),
               _ptr(g_m0), row, feat.data_ptr(), dl0.data_ptr(), dfeat.data_ptr(), B, P, K, F, ws.data_ptr(), ws.numel(), st)
        return
    C.call("ups_part_inject_bwd", g_inj.data_ptr(), feat.data_ptr(), hard.data_ptr(), dfeat.data_ptr(), dm.data_ptr(),
           B, P, K, F, ws.data_ptr(), ws.numel(), st)
    C.call("ups_part_softmax_bwd2", m0.data_ptr(), dm.data_ptr(), _ptr(g_m0), None, dl0.data_ptr(), B * P, K, st)


# The first convolutions folded into the sides (SURVEY 8f N4).  Shapes: feat [B,K,F], V [..,Co], G / dG [B,9,K,Co],
# masks [B,H,W,K], img [B,H,W,Cin].
def inject_conv_table_fwd(feat, V, G, st):
    B, K, F = feat.shape
    C.call("ups_inject_conv_table_fwd", feat.data_ptr(), V.data_ptr(), G.data_ptr(), B, K, F, V.shape[-1], st)


def inject_conv_table_bwd(dG, feat, V, dfeat, dV, st):
    B, K, F = feat.shape
    C.call("ups_inject_conv_table_bwd", dG.data_ptr(), feat.data_ptr(), V.data_ptr(), dfeat.data_ptr(), dV.data_ptr(),
           B, K, F, V.shape[-1], st)


def inject_conv_fwd(mask, G, bias, out, st):
    C.call("ups_inject_conv_fwd", mask.data_ptr(), G.data_ptr(), bias.data_ptr(), out.data_ptr(), *mask.shape, G.shape[-1],
           st)


def inject_conv_bwd(g_out, mask, G, probs, g_extra, dmask, dG, db, ws, st):
    C.call("ups_inject_conv_bwd", g_out.data_ptr(), mask.data_ptr(), G.data_ptr(), _ptr(probs), _ptr(g_extra),
           dmask.data_ptr(), dG.data_ptr(), db.data_ptr(), *mask.shape, G.shape[-1], ws.data_ptr(), ws.numel(), st)


def parts_conv_fwd(img, mask, V, bias, out, st):
    C.call("ups_parts_conv_fwd", img.data_ptr(), mask.data_ptr(), V.data_ptr(), bias.data_ptr(), out.data_ptr(),
           *mask.shape, img.shape[-1], V.shape[-1], st)


def parts_conv_bwd(g_out, img, mask, V, probs, g_extra, dmask, dV, db, ws, st):
    C.call("ups_parts_conv_bwd", g_out.data_ptr(), img.data_ptr(), mask.data_ptr(), V.data_ptr(), _ptr(probs),
           _ptr(g_extra), dmask.data_ptr(), dV.data_ptr(), db.data_ptr(), *mask.shape, img.shape[-1], V.shape[-1],
           ws.data_ptr(), ws.numel(), st)


def _on_device(fn):
    """Run a PartStep method with the step's device current: the C ABI launches on the device that is current on
    the calling thread, on the stream it is given, so both must be the device that owns the step's buffers."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapped


class PartStep:
    def __init__(self, batch_size, spatial_size, n_parts, local_app_size=64, n_views=3, use_tps=True,
                 views_grad=False, device="cuda", decode_bwd="auto", first_conv=0, encoder_conv=0, sample_offset=0,
                 tps_parameters=None, _planes=None):
        B, S, K, F, V = int(batch_size), int(spatial_size), int(n_parts), int(local_app_size), int(n_views)
        # sample_offset: global index of this step's first sample in the noise draw (forward(noise_seed=...)): a rank of a
        # data-parallel run that holds samples [o, o + B) of the global batch draws exactly what one GPU draws for them
        self.sample_offset = int(sample_offset)
        assert self.sample_offset >= 0
        self.B, self.S, self.K, self.F, self.V = B, S, K, F, V
        self.P = S * S
        # _planes (internal): part planes that really exist when this step runs a padded part count (see below)
        self.Kpl = K if _planes is None else int(_planes)
        self.use_tps = bool(use_tps) and V >= 2
        # tps_parameters: the ranges (tps.tps_parameters' keyword arguments) that forward(tps_seed=...) draws the warp from
        from . import configs
        from .tps import draw_scalars
        self.tps_parameters = dict(configs.CUB_TPS if tps_parameters is None else tps_parameters)
        self._tps_scalars = draw_scalars(**self.tps_parameters)
        self.views_grad = bool(views_grad)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise C.UpsError("PartStep needs a CUDA device: there is no CPU path")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.route, Kr = kernel_route(K, F, self.P, first_conv, encoder_conv)
        self.fused = self.route == "fused"
        # A part count that is not a power of two (the reference ships n_parts = 25, train_cub_subset_tps.yaml:132) runs on
        # the fused kernels of the next power of two Kp: logits padded with -inf, everything else with zeros.  exp_canon
        # maps -inf to exactly 0 and the canonical K-way sum is a pair tree over the zero-padded terms, so
        # probabilities, masks and labels are bit-identical to the K-part evaluation; padding planes of the part images
        # are neither written nor read (csrc: *_planes entry points).
        self.Kp = 0
        if self.route == "padded" and _planes is None:
            self.Kp = Kr
            self._inner = PartStep(B, S, self.Kp, F, n_views=V, use_tps=use_tps, views_grad=views_grad, device=self.device,
                                   decode_bwd=decode_bwd, sample_offset=sample_offset,
                                   tps_parameters=self.tps_parameters, _planes=K)
            self._init_padded()
            return
        # K4 variant: "tc" = persistent TMA + tcgen05/TMEM pipeline, "simt" = CUDA-core kernel
        tc_ok = self.fused and decode_bwd_tc_ok(K, F, self.P)
        assert decode_bwd in ("auto", "tc", "simt")
        if decode_bwd == "tc" and not tc_ok:
            raise C.UpsError("decode_bwd='tc' needs K in {16,32}, F == 64 and H*W % 128 == 0")
        self.decode_bwd = "tc" if (tc_ok and decode_bwd != "simt") else "simt"
        f32 = dict(dtype=torch.float32, device=self.device)
        e = torch.empty
        self.T = e(2 * B, 2, 11, **f32)
        # the warp parameters forward(tps_seed=...) draws (tps_drawn())
        self._tps_coord, self._tps_tv = e(2 * B, 8, 2, **f32), e(2 * B, 8, 2, **f32)
        self.warped = e(max(V, 2), B, S, S, 3, **f32) if self.use_tps else None
        self.m0, self.m1 = e(B, S, S, K, **f32), e(B, S, S, K, **f32)
        self.labels0 = e(B, S, S, dtype=torch.int64, device=self.device)
        self.parts = e(self.Kpl * B, S, S, 3, **f32) if not encoder_conv else None
        self.pooled = e(B, K, 3, **f32)
        # first_conv = Co > 0: the decode side ends in the decoder's first 3x3 convolution (h0 [B,S,S,Co]) instead of
        # the injected map; forward takes the filter (conv_V [3,3,F+K,Co], conv_b [Co]), backward g_h0
        self.Co = int(first_conv)
        if self.Co:
            self.inj = None
            self.h0 = e(B, S, S, self.Co, **f32)
            self.mh0c = e(B, S, S, K, **f32)
            self.G, self.dG = e(B, 9, K, self.Co, **f32), e(B, 9, K, self.Co, **f32)
            self.dV, self.db = e(3, 3, F + K, self.Co, **f32), e(self.Co, **f32)
            self.ws_ic = e(C.inject_conv_workspace_bytes(B, S, S, K, self.Co), dtype=torch.uint8, device=self.device)
            self._conv_V = None
        else:
            self.inj = e(B, S, S, F + K, **f32)
        # encoder_conv = Ce > 0: the encode side ends in the appearance encoder's first 3x3 convolution on the part images
        # (e0 [K*B,S,S,Ce], model.py:40,478) instead of the part images themselves; forward takes enc_V [3,3,3,Ce] and
        # enc_b [Ce], backward g_e0 in place of g_parts.  Neither `parts` nor `pooled` is formed (SURVEY 8f N4)
        self.Ce = int(encoder_conv)
        if self.Ce:
            assert not self.views_grad, "encoder_conv: the part images' convolution gives the image no gradient"
            self.parts = self.pooled = None
            self.e0 = e(K * B, S, S, self.Ce, **f32)
            self.mh1c = e(B, S, S, K, **f32)
            self.dVe, self.dbe = e(3, 3, 3, self.Ce, **f32), e(self.Ce, **f32)
            self.ws_pc = e(C.parts_conv_bwd_workspace_bytes(B, S, S, K, self.Ce), dtype=torch.uint8, device=self.device)
            self._enc_V = None
        self.dl0, self.dl1 = e(B, S, S, K, **f32), e(B, S, S, K, **f32)
        self.dfeat = e(B, K, F, **f32)
        nws = C.workspace_bytes(C.OP_STEP, B, self.P, K, F)
        self.ws = e(nws, dtype=torch.uint8, device=self.device)
        if self.views_grad:
            self.dimg1 = e(B, S, S, 3, **f32)
            self.dviews = e(max(V, 2), B, S, S, 3, **f32)
        self.mh0 = self.mh1 = self.dm = self.dm2 = self.dfm = None   # the generic kernels' masks and scratch
        if not self.fused:
            self.mh0, self.mh1 = e(B, S, S, K, **f32), e(B, S, S, K, **f32)
            self.dm = e(B, S, S, K, **f32)
            self.dm2 = e(B, S, S, K, **f32)
            self.dfm = e(B, S, S, 3, **f32)
        # K1 and K3 in one launch (csrc/step_fwd_fused.cu); UPS_FUSE_FWD=0 keeps them as two kernels
        self.fuse_fwd = (self.fused and self.use_tps and not self.Co and not self.Ce and K in (8, 16, 32) and F in (16, 32, 64)
                         and os.environ.get("UPS_FUSE_FWD", "1") != "0")
        self.before_params = None   # optional callable, invoked in forward just before the first kernel that depends on
        #                             the surrounding model's parameters (logits / features)
        self._labels_u8 = None
        self._views_f32 = None   # allocated on first use: fp32 copy of uint8 views (data.py:134 on the device)
        self._img1 = None
        self._warped = None
        self._feat = None
        self._coord = None

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_tps(self, coord, t_vector, tps_seed):
        """forward's warp arguments: given coord and t_vector, or tps_seed alone."""
        if tps_seed is None:
            if self.use_tps and (coord is None or t_vector is None):
                raise ValueError("PartStep.forward: pass coord and t_vector, or tps_seed to draw them on the device")
            return
        if coord is not None or t_vector is not None:
            raise ValueError("PartStep.forward: pass coord and t_vector, or tps_seed, not both")
        if not self.use_tps:
            raise ValueError("PartStep.forward: tps_seed needs a step with use_tps")
        if isinstance(tps_seed, torch.Tensor):
            if tps_seed.dtype != torch.int64 or tps_seed.numel() != 1 or tps_seed.device != self.device \
                    or not tps_seed.is_contiguous():
                raise C.UpsError("PartStep: a device tps_seed is a contiguous one-element int64 tensor on the step's device")
        else:
            _seed_i64(tps_seed)
            if torch.cuda.is_current_stream_capturing():
                raise C.UpsError("PartStep: an int tps_seed is frozen into a captured CUDA graph (every replay would draw "
                                 "the same warp); pass the seed as a one-element int64 CUDA tensor")

    def _tps_solve(self, coord, t_vector, tps_seed, st):
        """The 11x11 systems of the 2B warps into self.T: of the given coord / t_vector, or of the warp drawn from
        tps_seed (view v of global sample sample_offset + b in row v * B + b) into the step's own buffers, in the same
        one launch.  Returns the coord the warp uses."""
        B = self.B
        if tps_seed is None:
            assert tuple(coord.shape) == (2 * B, 8, 2) and tuple(t_vector.shape) == (2 * B, 8, 2)
            C.call("ups_tps_solve", coord.data_ptr(), t_vector.data_ptr(), self.T.data_ptr(), 2 * B, st)
            return coord
        C.call("ups_tps_draw_solve_dseed" if isinstance(tps_seed, torch.Tensor) else "ups_tps_draw_solve",
               _seed_arg(tps_seed), self.sample_offset, B, 2, *self._tps_scalars, self._tps_coord.data_ptr(), None, None,
               None, None, None, self._tps_tv.data_ptr(), self.T.data_ptr(), st)
        return self._tps_coord

    def tps_drawn(self):
        """The warp the last forward(tps_seed=...) drew: dict(coord, t_vector) [2B,8,2], views of the step's buffers.
        forward(views, coord, t_vector, ...) with copies of them computes the same bits."""
        if self.Kp:
            return self._inner.tps_drawn()
        return dict(coord=self._tps_coord, t_vector=self._tps_tv)

    def _noise(self, noise_seed, noise_level):
        """The launchers' noise value of forward(noise_seed=, noise_level=): None, or (seed, sample_offset, noise_level)."""
        return None if noise_seed is None else (_seed_i64(noise_seed), self.sample_offset, float(noise_level))

    # ------------------------------------------------------------------ padded part count (K -> Kp)
    def _init_padded(self):
        B, S, K, F, Kp = self.B, self.S, self.K, self.F, self.Kp
        f32 = dict(dtype=torch.float32, device=self.device)
        inner = self._inner
        self.fused, self.fuse_fwd, self.decode_bwd, self.Co = True, inner.fuse_fwd, inner.decode_bwd, 0
        # padded inputs, pad regions written once: -inf for logits, 0 for everything else
        self._l0p = torch.full((B, S, S, Kp), float("-inf"), **f32)
        self._l1p = torch.full((B, S, S, Kp), float("-inf"), **f32)
        self._featp = torch.zeros(B, Kp, F, **f32)
        self._g_injp = torch.zeros(B, S, S, F + Kp, **f32)
        self._g_m0p, self._g_m1p = torch.zeros(B, S, S, Kp, **f32), torch.zeros(B, S, S, Kp, **f32)
        self._g_pooledp = torch.zeros(B, Kp, 3, **f32)
        # outputs are VIEWS of the inner step's padded buffers (row pitch Kp floats): nothing is copied back
        self.m0, self.m1 = inner.m0[..., :K], inner.m1[..., :K]
        self.inj = inner.inj[..., :F + K]
        self.dl0, self.dl1 = inner.dl0[..., :K], inner.dl1[..., :K]
        self.pooled, self.dfeat = inner.pooled[:, :K], inner.dfeat[:, :K]
        self.labels0, self.parts, self.warped = inner.labels0, inner.parts, inner.warped
        self._labels_u8 = None

    def pitched_inputs(self):
        """Padded part count only: views [..., :K] of the step's internal row-pitched input buffers (l0, l1, g_inj, g_m0,
        g_m1).  A producer that writes its logits / cotangents into these (row pitch Kp floats instead of K) hands them
        to forward / backward without any copy; contiguous tensors are accepted as well and are copied into the buffers."""
        assert self.Kp, "pitched_inputs() is for part counts that are not a power of two"
        K, F = self.K, self.F
        return dict(l0=self._l0p[..., :K], l1=self._l1p[..., :K], g_inj=self._g_injp[..., :F + K],
                    g_m0=self._g_m0p[..., :K], g_m1=self._g_m1p[..., :K])

    def _arg(self, t, buf):
        """(tensor to hand to the kernel, its row length): the pitched buffer itself when `t` is its view, else the
        caller's contiguous [.,K] tensor, which the kernels read in place."""
        if t.data_ptr() == buf.data_ptr() and t.stride() == buf.stride():
            return buf, self.Kp
        assert t.is_contiguous() and t.shape[-1] == self.K, "pass a contiguous tensor or the view from pitched_inputs()"
        return t, self.K

    def _into(self, t, buf, n_cols, fill, st):
        """t [.., n_cols] -> the row-pitched buffer `buf` [.., pitch]; no-op when t already is the buffer's view."""
        if t.data_ptr() == buf.data_ptr() and t.stride() == buf.stride() and t.shape[-1] == n_cols:
            return
        assert t.is_contiguous(), "pass a contiguous tensor or the view from pitched_inputs()"
        n_rows = t.numel() // n_cols
        C.call("ups_copy_rows", t.data_ptr(), n_cols, buf.data_ptr(), buf.shape[-1], n_rows, n_cols,
               buf.shape[-1] - n_cols, fill, st)

    @_on_device
    def _forward_padded(self, views, coord, t_vector, l0, l1, feat, noise_seed=None, noise_level=1.0, tps_seed=None):
        B, S, K, F, P, Kp = self.B, self.S, self.K, self.F, self.P, self.Kp
        st = self._stream()
        assert feat.is_contiguous()
        assert tuple(l0.shape) == (B, S, S, K) and tuple(l1.shape) == (B, S, S, K) and tuple(feat.shape) == (B, K, F)
        # logits: a contiguous [.,K] tensor is read in place by the kernels (row length K, parts >= K are -inf); the
        # pitched view of pitched_inputs() already is the padded buffer
        a0, n0 = self._arg(l0, self._l0p)
        a1, n1 = self._arg(l1, self._l1p)
        # feat [B,K,F] -> [B,Kp,F]: per sample the first K*F floats of the padded block (the rest stays zero)
        C.call("ups_copy_rows", feat.data_ptr(), K * F, self._featp.data_ptr(), Kp * F, B, K * F, 0, 0.0, st)
        o = self._inner.forward(views, coord, t_vector, a0, a1, self._featp, rows=dict(l0=n0, l1=n1), noise_seed=noise_seed,
                                noise_level=noise_level, tps_seed=tps_seed)
        self._feat, self._img1 = feat, self._inner._img1
        return dict(warped=o["warped"], m0=self.m0, m1=self.m1, labels0=self.labels0, parts=self.parts, pooled=self.pooled,
                    inj=self.inj)

    @_on_device
    def _backward_padded(self, g_inj, g_parts, g_pooled, g_m0, g_m1, g_warped):
        B, S, K, F, P, Kp = self.B, self.S, self.K, self.F, self.P, self.Kp
        st = self._stream()
        assert tuple(g_inj.shape) == (B, S, S, F + K) and tuple(g_parts.shape) == (K * B, S, S, 3)
        self._into(g_inj, self._g_injp, F + K, 0.0, st)
        gm0 = gm1 = gpl = None
        n0 = n1 = Kp
        if g_m0 is not None:
            gm0, n0 = self._arg(g_m0, self._g_m0p)
        if g_m1 is not None:
            gm1, n1 = self._arg(g_m1, self._g_m1p)
        if g_pooled is not None:
            C.call("ups_copy_rows", g_pooled.data_ptr(), K * 3, self._g_pooledp.data_ptr(), Kp * 3, B, K * 3, 0, 0.0, st)
            gpl = self._g_pooledp
        o = self._inner.backward(self._g_injp, g_parts, gpl, gm0, gm1, g_warped, rows=dict(g_m0=n0, g_m1=n1))
        out = dict(dl0=self.dl0, dl1=self.dl1, dfeat=self.dfeat)
        if "dviews" in o:
            out["dviews"] = o["dviews"]
        return out

    # ------------------------------------------------------------------ forward
    def forward(self, views, coord, t_vector, l0, l1, feat, conv_V=None, conv_b=None, enc_V=None, enc_b=None, rows=None,
                noise_seed=None, noise_level=1.0, tps_seed=None):
        """views [V,B,S,S,3] (view0, view1[, view0_target]), fp32 in [-1, 1] or the dataset's uint8
        (normalised on the device exactly as cub/code/data/data.py:134 does on the host); coord,
        t_vector [2B,8,2] from make_input_tps_param; l0, l1 [B,S,S,K]; feat [B,K,F].  Returns a dict
        of views into the step's persistent output buffers.

        noise_seed (an integer in [0, 2**64)): the reference's training step, which samples its logits
        (MeanFieldDistribution.sample, model.py:420-421): l0 and l1 are the MEANS and the kernels use
        l = mean + noise_level * eps, eps ~ N(0,1) drawn in registers right after the load (draw 0 for l0, 1 for l1, global
        pixel (sample_offset + b) * S*S + p; csrc/canon_math.cuh).  No extra pass and no extra launch.  The sampled logits
        are not written (the reference keeps them as m0_logits / m1_logits): ups_normal_philox_fwd(seed, draw,
        sample_offset * S*S, B*S*S, K) gives eps bit for bit, and ops.mean_field_sample(mean, eps, noise_level) the logits
        (nn.MeanFieldDistribution(mean).sample(noise_level, seed=..., draw=..., sample_offset=...) does both).
        backward is unchanged: d l / d mean is the identity, so dl0 / dl1 are the gradients of the means.
        noise_seed=None is the noise-free step (l0, l1 are the logits), with the same launches as always.

        On the fused path K1 (TPS warp) and K3 (decode side) are independent and run as ONE launch with interleaved
        CTAs (ups_step_warp_decode_fwd): the warp's arithmetic hides under the decode side's memory stream.
        forward_warp / forward_parts are the same step as two calls (K1 | K2, K3) for callers that have the views
        before the logits.

        tps_seed (an int in [0, 2**64), or a one-element int64 CUDA tensor read by the kernel, which a captured CUDA graph
        needs; pass coord = t_vector = None): the warp parameters are drawn on the device instead, from the ranges of
        the constructor's tps_parameters, as tps.tps_parameters(2B, seed=tps_seed, sample_offset=sample_offset, views=2)
        draws them.  The draw runs in the launch that otherwise solves the given warp, so the step issues as many
        launches as with given coord; tps_drawn() returns the drawn coord / t_vector."""
        self._check_tps(coord, t_vector, tps_seed)
        if self.Kp:
            return self._forward_padded(views, coord, t_vector, l0, l1, feat, noise_seed, noise_level, tps_seed)
        # rows (internal, padded part counts): row lengths of l0 / l1 when they are read in place ({"l0": 25, "l1": 25})
        if self.fuse_fwd:
            return self._forward_fused(views, coord, t_vector, l0, l1, feat, rows, self._noise(noise_seed, noise_level),
                                       tps_seed)
        self.forward_warp(views, coord, t_vector, tps_seed)
        return self.forward_parts(l0, l1, feat, conv_V, conv_b, enc_V, enc_b, rows, noise_seed, noise_level)

    @_on_device
    def _forward_fused(self, views, coord, t_vector, l0, l1, feat, rows=None, nz=None, tps_seed=None):
        B, S, K, F, P, V = self.B, self.S, self.K, self.F, self.P, self.V
        st = self._stream()
        views = self._ingest(views, st)
        r0, r1 = (rows or {}).get("l0", K), (rows or {}).get("l1", K)
        assert l0.is_contiguous() and l1.is_contiguous() and feat.is_contiguous()
        assert tuple(l0.shape) == (B, S, S, r0) and tuple(l1.shape) == (B, S, S, r1) and tuple(feat.shape) == (B, K, F)
        coord = self._tps_solve(coord, t_vector, tps_seed, st)
        if self.before_params is not None:
            self.before_params()     # data-parallel wrapper: wait for the averaged gradients (the TPS solve needs none)
        call_rows("ups_step_warp_decode_fwd_rows", nz, views.data_ptr(), views[2].data_ptr() if V > 2 else None,
                  coord.data_ptr(), self.T.data_ptr(), self.warped.data_ptr(), self.warped[2].data_ptr() if V > 2 else None,
                  2 * B, B if V > 2 else 0, S, l0.data_ptr(), r0, feat.data_ptr(), self.m0.data_ptr(),
                  self.labels0.data_ptr(), self.inj.data_ptr(), B, K, F, st)
        self._warped, self._coord = self.warped, coord
        img1 = self.warped[1]
        self._img1, self._feat = img1, feat
        encode_fwd(self.route, nz, l1, img1, self.m1, self.parts, self.pooled, None, self.ws, B, P, K, r1, self.Kpl, st)
        return dict(warped=self.warped, m0=self.m0, m1=self.m1, labels0=self.labels0, parts=self.parts,
                    pooled=self.pooled, inj=self.inj)

    @_on_device
    def labels_u8(self):
        """labels0 narrowed to uint8 on the device (n_parts <= 255): the label map a host-side consumer reads back,
        one byte per pixel instead of tf.argmax's eight."""
        assert self.K <= 255
        if self.Kp:
            return self._inner.labels_u8()
        if self._labels_u8 is None:
            self._labels_u8 = torch.empty(self.labels0.shape, dtype=torch.uint8, device=self.device)
        C.call("ups_labels_i64_to_u8", self.labels0.data_ptr(), self._labels_u8.data_ptr(), self.labels0.numel(),
               self._stream())
        return self._labels_u8

    def _ingest(self, views, st):
        B, S, V = self.B, self.S, self.V
        if views.dtype == torch.uint8:
            assert views.is_contiguous() and tuple(views.shape) == (V, B, S, S, 3), list(views.shape)
            if self._views_f32 is None:
                self._views_f32 = torch.empty(V, B, S, S, 3, dtype=torch.float32, device=self.device)
            C.call("ups_views_u8_to_f32", views.data_ptr(), self._views_f32.data_ptr(), views.numel(), st)
            views = self._views_f32
        assert views.is_contiguous() and tuple(views.shape) == (V, B, S, S, 3), list(views.shape)
        return views

    @_on_device
    def forward_warp(self, views, coord, t_vector, tps_seed=None):
        """K1: the TPS equivariance warp of the views (model.py:282-311).  Returns the warped views [V,B,S,S,3].
        tps_seed: draw the warp on the device (see forward)."""
        B, S, V = self.B, self.S, self.V
        st = self._stream()
        views = self._ingest(views, st)
        if self.use_tps:
            coord = self._tps_solve(coord, t_vector, tps_seed, st)
            if V > 2:  # the target view shares view0's warp (model.py:306-309): one launch, shared grid
                C.call("ups_tps_warp_pair_fwd", views.data_ptr(), views[2].data_ptr(), coord.data_ptr(),
                       self.T.data_ptr(), self.warped.data_ptr(), self.warped[2].data_ptr(), 2 * B, B, S, S, 3, S, S, st)
            else:
                C.call("ups_tps_warp_fwd", views.data_ptr(), coord.data_ptr(), self.T.data_ptr(), None, None,
                       self.warped.data_ptr(), None, 2 * B, S, S, 3, S, S, st)
            self._warped = self.warped
            self._coord = coord
        else:
            self._warped = views
        return self._warped

    @_on_device
    def forward_parts(self, l0, l1, feat, conv_V=None, conv_b=None, enc_V=None, enc_b=None, rows=None, noise_seed=None,
                      noise_level=1.0):
        """K2 (encode side: l1, warped view 1) and K3 (decode side: l0, feat) on the current stream.  noise_seed /
        noise_level: l0, l1 are means, sampled inside the kernels (see forward)."""
        B, S, K, F, P = self.B, self.S, self.K, self.F, self.P
        st = self._stream()
        nz = self._noise(noise_seed, noise_level)
        r0, r1 = (rows or {}).get("l0", K), (rows or {}).get("l1", K)
        assert (r0 == K and r1 == K) or (self.fused and not self.Co and not self.Ce), "in-place rows need the fused kernels"
        assert l0.is_contiguous() and l1.is_contiguous() and feat.is_contiguous()
        assert tuple(l0.shape) == (B, S, S, r0) and tuple(l1.shape) == (B, S, S, r1) and tuple(feat.shape) == (B, K, F)
        if self.Co:
            assert conv_V is not None and conv_b is not None, "first_conv: pass conv_V [3,3,F+K,Co] and conv_b [Co]"
            assert tuple(conv_V.shape) == (3, 3, F + K, self.Co) and tuple(conv_b.shape) == (self.Co,)
            assert conv_V.is_contiguous() and conv_b.is_contiguous()
            self._conv_V = conv_V
        warped = self._warped
        img1 = warped[1]
        self._img1, self._feat = img1, feat
        if self.Ce:
            assert enc_V is not None and enc_b is not None, "encoder_conv: pass enc_V [3,3,3,Ce] and enc_b [Ce]"
            assert tuple(enc_V.shape) == (3, 3, 3, self.Ce) and tuple(enc_b.shape) == (self.Ce,)
            assert enc_V.is_contiguous() and enc_b.is_contiguous()
            self._enc_V = enc_V
            part_softmax_fwd(nz, 1, l1, self.m1, None, self.mh1c, B, P, K, st)
            parts_conv_fwd(img1, self.mh1c, enc_V, enc_b, self.e0, st)
        else:
            encode_fwd(self.route, nz, l1, img1, self.m1, self.parts, self.pooled, self.mh1, self.ws, B, P, K, r1, self.Kpl,
                       st)
        if self.Co:
            part_softmax_fwd(nz, 0, l0, self.m0, self.labels0, self.mh0c, B, P, K, st)
            inject_conv_table_fwd(feat, conv_V, self.G, st)
            inject_conv_fwd(self.mh0c, self.G, conv_b, self.h0, st)
        else:
            decode_fwd(self.route, nz, l0, feat, self.m0, self.labels0, self.inj, self.mh0, B, P, K, F, r0, st)
        out = dict(warped=warped, m0=self.m0, m1=self.m1, labels0=self.labels0)
        if self.Ce:
            out["e0"] = self.e0
        else:
            out["parts"], out["pooled"] = self.parts, self.pooled
        if self.Co:
            out["h0"] = self.h0
        else:
            out["inj"] = self.inj
        return out

    # ------------------------------------------------------------------ backward
    def backward(self, g_inj, g_parts, g_pooled=None, g_m0=None, g_m1=None, g_warped=None, rows=None):
        """Cotangents: g_inj [B,S,S,F+K] (with first_conv: g_h0 [B,S,S,Co] in its place), g_parts [K*B,S,S,3]
        (part-major), g_pooled [B,K,3], g_m0/g_m1 [B,S,S,K] (from the mask losses), g_warped [V,B,S,S,3]
        (views_grad only).  Returns dict(dl0, dl1, dfeat[, dV, db][, dviews]).  After a forward with noise_seed, dl0 / dl1
        are the gradients of the means (the sample is mean + a constant).

        = backward_decode (K4: dl0, dfeat — what the appearance encoder's backward needs) followed by
        backward_encode (K5 [, K6]: dl1 [, dviews])."""
        if self.Kp:
            return self._backward_padded(g_inj, g_parts, g_pooled, g_m0, g_m1, g_warped)
        out = self.backward_decode(g_inj, g_m0, (rows or {}).get("g_m0"))
        out.update(self.backward_encode(g_parts, g_pooled, g_m1, g_warped, (rows or {}).get("g_m1")))
        return out

    @_on_device
    def backward_decode(self, g_inj, g_m0=None, gm_row=None):
        """K4: autodiff of the decode side.  g_inj, g_m0 -> dl0 [B,S,S,K], dfeat [B,K,F] [, dV, db]."""
        B, S, K, F, P = self.B, self.S, self.K, self.F, self.P
        st = self._stream()
        feat = self._feat
        if self.Co:
            assert tuple(g_inj.shape) == (B, S, S, self.Co), list(g_inj.shape)
            inject_conv_bwd(g_inj, self.mh0c, self.G, self.m0, g_m0, self.dl0, self.dG, self.db, self.ws_ic, st)
            inject_conv_table_bwd(self.dG, feat, self._conv_V, self.dfeat, self.dV, st)
        else:
            decode_bwd(self.route, self.decode_bwd == "tc", g_inj, g_m0, self.m0, self.mh0, feat, self.dl0, self.dfeat,
                       self.dm, self.ws, B, P, K, F, gm_row or K, st)
        out = dict(dl0=self.dl0, dfeat=self.dfeat)
        if self.Co:
            out["dV"], out["db"] = self.dV, self.db
        return out

    @_on_device
    def backward_encode(self, g_parts, g_pooled=None, g_m1=None, g_warped=None, gm_row=None):
        """K5 (autodiff of the encode side: dl1 [, dimg1]) and, with views_grad, K6 (TPS backward: dviews)."""
        B, S, K, P, V = self.B, self.S, self.K, self.P, self.V
        st = self._stream()
        img1 = self._img1
        if self.Ce:
            assert tuple(g_parts.shape) == (K * B, S, S, self.Ce), list(g_parts.shape)      # g_e0 in the place of g_parts
            parts_conv_bwd(g_parts, img1, self.mh1c, self._enc_V, self.m1, g_m1, self.dl1, self.dVe, self.dbe, self.ws_pc, st)
            return dict(dl1=self.dl1, dVe=self.dVe, dbe=self.dbe)
        encode_bwd(self.route, g_parts, g_pooled, g_m1, img1, self.m1, self.mh1, self.dl1,
                   self.dimg1 if self.views_grad else None, self.dm, self.dm2, self.dfm, B, P, K, gm_row or K, self.Kpl, st)
        out = dict(dl1=self.dl1)
        if self.views_grad:
            if self.use_tps:
                # cotangent of the warped views: g_warped (+ dimg1 on view 1), formed inside K6 (never materialised)
                coord, gw = self._coord, g_warped
                if gw is not None:
                    assert gw.is_contiguous() and tuple(gw.shape) == (max(V, 2), B, S, S, 3), list(gw.shape)
                pair = V > 2 and gw is not None
                C.call("ups_tps_warp_bwd_sum", _ptr(gw), gw[2].data_ptr() if pair else None, self.dimg1.data_ptr(), B, B,
                       coord.data_ptr(), self.T.data_ptr(), self.dviews.data_ptr(),
                       self.dviews[2].data_ptr() if pair else None, 2 * B, B, S, S, 3, S, S, st)
                if V > 2 and gw is None:
                    C.call("ups_views_cotangent", None, None, self.dviews[2].data_ptr(), 1, 0, B * P * 3, st)   # zeros
            else:
                C.call("ups_views_cotangent", _ptr(g_warped), self.dimg1.data_ptr(), self.dviews.data_ptr(), max(V, 2), 1,
                       B * P * 3, st)
            out["dviews"] = self.dviews
        return out

    # kernels enqueued by one forward+backward (bench.py's gpu_launches is counted, not assumed)
    def algorithmic_bytes_per_image(self):
        """SURVEY.md 8d / BASELINE.md 4: 4*P*(6V + 18K + 2F + 5 [+6V]) + 12*K*F + 8*K*C."""
        V = self.V if self.use_tps else 0
        per_px = 6 * V + 18 * self.K + 2 * self.F + 5 + (6 * V if self.views_grad else 0)
        return 4 * self.P * per_px + 12 * self.K * self.F + 8 * self.K * 3
