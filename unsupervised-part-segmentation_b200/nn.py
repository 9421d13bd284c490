"""Drop-in for the part-map helpers of the reference's `nips19.nn` module
(cub/code/nn.py == pennaction/code/nn.py; deepfashion/code/nn.py): same names, argument
order and defaults; torch CUDA tensors (NHWC, fp32) instead of TF graph tensors."""
import torch

from . import ops


def softmax(x, spatial=False):
    """cub/code/nn.py:58-62 — K-way softmax over the last axis (spatial=True: over H*W)."""
    if spatial:
        return spatial_softmax(x)
    return ops.part_softmax(x)


def spatial_softmax(features):
    """cub/code/nn.py:65-71 — [N,H,W,C] -> softmax over H*W for every (n, c)."""
    assert features.dim() == 4, list(features.shape)
    return ops.spatial_softmax(features)


def _to_last(y, axis):
    axis = axis % y.dim()
    return (y, None) if axis == y.dim() - 1 else (y.movedim(axis, -1).contiguous(), axis)


def hard_max(y, axis):
    """cub/code/nn.py:134-136 — float(y == reduce_max(y, axis, keep_dims=True)); every tied
    maximum is marked.  Not differentiable (tf.equal)."""
    yl, moved = _to_last(y.detach(), axis)
    out = ops.hard_max(yl)
    return out if moved is None else out.movedim(-1, moved)


def straight_through_estimator(y_hard, y):
    """cub/code/nn.py:154-168 — tf.stop_gradient(y_hard - y) + y."""
    return ops.straight_through(y_hard.detach(), y)


def hard_max_straight_through(y, axis):
    """cub/code/nn.py:117-131 (deprecated in the reference in favour of the two calls)."""
    return straight_through_estimator(hard_max(y, axis), y)


def apply_partwise(input_, func):
    """cub/code/nn.py:81-113 — [b,h,w,parts,f] -> part-major [parts*b,h,w,f] -> func ->
    [b,h_out,w_out,parts,c_out]."""
    b, h, w, parts, f = input_.shape
    x = ops.partwise_fold(input_)
    y = func(x)
    assert y.dim() == 4 and y.shape[0] == parts * b, list(y.shape)
    return ops.partwise_unfold(y, parts)


def mask2hotmask(mask, n_parts):
    """cub/code/nn.py:2086-2089 — one_hot(argmax(mask, 3), n_parts)."""
    return ops.one_hot(ops.argmax(mask.detach()), n_parts)


def argmax(y, axis=3):
    """tf.argmax(y, 3) as used at cub/code/SB_model48i/model.py:447,465,470 — int64, first index."""
    yl, _ = _to_last(y.detach(), axis)
    return ops.argmax(yl)


def unpool_features_gathered(feature_vectors, mask):
    """cub/code/nn.py:2469-2487 — feature_vectors [B,parts,F], integer mask [B,h,w] -> [B,h,w,F]."""
    bs, h, w = mask.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs, fshape
    return ops.part_gather(feature_vectors, mask)


def draw_rect(center, height, width, shape):
    """tfutils.draw_rect as called at cub/code/SB_model48i/model.py:442 — center [N,2] integer (row, column), rectangle
    height x width, shape = [h, w, 1] -> [N,h,w,1] of 0/1.  `tfutils` is not vendored with the reference; the
    convention (rows [cy - height//2, cy - height//2 + height), same for columns, clipped) is documented in
    include/ups_b200.h."""
    h, w = int(shape[0]), int(shape[1])
    return ops.draw_rect(center, int(height), int(width), h, w)[..., None]


def patch_masks(mask_hard, patch_size, gamma=3.0):
    """cub/code/SB_model48i/model.py:437-445: the square patch around each part's centre of mass —
    softmax(spatial=True) of gamma * mask, probs_to_mu_sigma, centres cast to int pixels (truncation, as tf.cast),
    draw_rect, back to [N,h,w,P].  No gradient (tf.stop_gradient at the call site)."""
    N, h, w, P = mask_hard.shape
    with torch.no_grad():
        corrected = softmax(mask_hard * gamma, spatial=True)
        mu, _ = probs_to_mu_sigma(corrected, torch.ones(N, P, device=mask_hard.device))
        centers = (mu.reshape(N * P, 2) * h / 2.0 + h / 2.0).to(torch.int32)
        rect = draw_rect(centers, patch_size, patch_size, [h, w, 1])
        return rect.reshape(N, P, h, w).permute(0, 2, 3, 1).contiguous()


def probs_to_mu_sigma(probs, scaling_factor):
    """cub/code/nn.py:1541-1587 — per-part mean (y, x) and 2x2 covariance of the [b,h,w,k] densities on
    the linspace(-1, 1) grid; scaling_factor [b,k].  Returns (mu [b,k,2], sigma [b,k,2,2])."""
    bn, h, w, nk = probs.shape
    sf = scaling_factor.reshape(bn, nk)
    mu, sigma, _ = ops.mask_moments(probs, sf)
    return mu, sigma


# ------------------------------------------------------------------ mask priors and sampling (SURVEY.md 8f N2/N3)
def mumford_shah(x, alpha, lambda_):
    """cub/code/nn.py:1381-1386 — (r, smoothness_cost, contour_cost) of the finite-difference energy
    g = |tf_grad(x)|^2 (nn.py:1357-1378), each [b,h,w,k]."""
    assert x.dim() == 4, list(x.shape)
    return ops.mumford_shah(x, float(alpha), float(lambda_))


def mumford_shah_sums(x, alpha, lambda_):
    """The four spatial sums cub/code/SB_model48i/model.py:744-769 squares: [b,4,k] = sum over (h,w) of
    (r, smoothness_cost, contour_cost, x), in one pass over x and without the three [b,h,w,k] maps."""
    assert x.dim() == 4, list(x.shape)
    return ops.mumford_shah_sums(x, float(alpha), float(lambda_))


def edge_set(x, alpha, lambda_):
    """cub/code/nn.py:1389-1392."""
    assert x.dim() == 4, list(x.shape)
    return ops.edge_set(x.detach(), float(alpha), float(lambda_))


class MeanFieldDistribution(object):
    """cub/code/nn.py:1395-1457 — the distribution object on the part logits (model.py:413-421).  TF's RNG stream is not
    reproducible; `sample` takes its N(0,1) draw from one of three sources:
      eps=...       the caller's tensor;
      seed=...      the project's counter-based draw (csrc/canon_math.cuh), generated on the device: a pure function of
                    (seed, draw, global pixel, part), so it regenerates bit for bit what PartStep.forward(noise_seed=seed)
                    drew inside the step (draw 0 for l0, 1 for l1; sample_offset = global index of sample 0);
      neither       torch.randn with `generator`."""

    def __init__(self, parameters, dim, stochastic=True):
        self.parameters = parameters
        self.dim = dim
        self.stochastic = stochastic
        ps = list(self.parameters.shape)
        assert len(ps) == 4
        self.batch_size = ps[0]
        self.event_axes = [1, 2, 3]
        self.mean = self.parameters
        self.shape = ps
        self._priors = None

    @staticmethod
    def n_parameters(dim):
        return dim

    def _philox_args(self, seed, draw, sample_offset):
        assert self.mean.dim() == 4
        B, H, W, K = self.shape
        return ops._seed_i64(seed), int(draw), int(sample_offset) * H * W, B * H * W, K

    def sample(self, noise_level=1.0, eps=None, generator=None, seed=None, draw=0, sample_offset=0):
        if not self.stochastic:
            return self.mean
        if eps is None and seed is not None:
            s, d, off, n, K = self._philox_args(seed, draw, sample_offset)
            eps = ops.normal_philox(s, d, off, n, K, self.mean.device).view(self.shape)
        if eps is None:
            eps = torch.randn(self.shape, generator=generator, device=self.mean.device, dtype=torch.float32)
        return ops.mean_field_sample(self.mean, eps, float(noise_level))

    def sample_softmax(self, noise_level=1.0, eps=None, generator=None, seed=None, draw=0, sample_offset=0):
        """softmax(sample()) in one pass (cub/code/SB_model48i/model.py:420-430): -> (logits, probs, labels, hard)
        with hard = straight_through_estimator(hard_max(probs, 3), probs).  With `seed` the draw is made in registers."""
        if not self.stochastic:
            probs, labels, hard = ops.part_softmax_full(self.mean)
            return self.mean, probs, labels, hard
        if eps is None and seed is not None:
            s, d, off, _, _ = self._philox_args(seed, draw, sample_offset)
            return ops.part_softmax_sampled_philox(self.mean, s, d, off, float(noise_level))
        if eps is None:
            eps = torch.randn(self.shape, generator=generator, device=self.mean.device, dtype=torch.float32)
        return ops.part_softmax_sampled(self.mean, eps, float(noise_level))

    def _all(self):
        if self._priors is None:
            self._priors = ops.logit_priors(self.mean)      # one pass yields the three energies
        return self._priors

    def kl(self, other=None):
        if other is not None:
            raise NotImplementedError("Only KL to standard normal is implemented.")
        return self._all()[0]

    def kl_improper_gmrf(self):
        return self._all()[1]

    def kl_tv(self):
        return self._all()[2]

    def kl_mumford_sha(self, alpha, lambda_):
        r, _, _ = mumford_shah(self.mean, alpha, lambda_)
        return r.sum(dim=self.event_axes).mean()


def mask2rgb(mask, make_hot=True, colors=None):
    """cub/code/nn.py:2067-2083 — [b,h,w,k] -> [b,h,w,3] in [-1,1].  `colors` [k,3] in [0,1] replaces the reference's
    make_mask_colors (matplotlib's inferno LUT, not available here): default = an evenly spaced grey ramp."""
    n_parts = mask.shape[3]
    if colors is None:
        colors = torch.linspace(0, 1, n_parts, dtype=torch.float64)[:, None].repeat(1, 3)
    table = ((torch.as_tensor(colors).to(torch.float64).cpu() - 0.5) * 2).to(torch.float32).to(mask.device)
    return ops.mask2rgb(mask.detach(), table, bool(make_hot))
