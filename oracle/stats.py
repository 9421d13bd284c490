"""TEST INFRASTRUCTURE — CPU restatement of the mask statistics the training step computes on the
part probabilities (SURVEY.md 8f N1/N2).  Pinned against tests/golden/stats.npz (the reference's
function bodies run under tf1_shim)."""
import torch


def probs_to_mu_sigma(probs, scaling_factor):
    """cub/code/nn.py:1541-1587.  probs [b,h,w,k]; scaling_factor [b,k] -> mu [b,k,2] (y, x),
    sigma [b,k,2,2].  Evaluated in the dtype and on the device of `probs` (float64 gives the tests' exact reference)."""
    bn, h, w, nk = probs.shape
    y_t = torch.linspace(-1.0, 1.0, h, dtype=probs.dtype, device=probs.device).reshape(h, 1).repeat(1, w)
    x_t = torch.linspace(-1.0, 1.0, w, dtype=probs.dtype, device=probs.device).reshape(1, w).repeat(h, 1)
    meshgrid = torch.stack([y_t, x_t], dim=-1)                               # [h,w,2]
    mu = torch.einsum("ijl,aijk->akl", meshgrid, probs)
    mu_out_prod = torch.einsum("akm,akn->akmn", mu, mu)
    mesh_out_prod = torch.einsum("ijm,ijn->ijmn", meshgrid, meshgrid)
    stddev = torch.einsum("ijmn,aijk->akmn", mesh_out_prod, probs) - mu_out_prod
    sigma = (scaling_factor ** 2)[..., None, None] * stddev
    mu = mu * scaling_factor[..., None]
    return mu, sigma


def categorical_kl(probs):
    """cub/code/SB_model48i/model.py:21-25."""
    k = float(probs.shape[-1])
    logkp = torch.log(k * probs + 1e-20)
    kl = (probs * logkp).sum(dim=-1)
    return kl.mean()


def draw_rect(centers, ph, pw, H, W):
    """tfutils.draw_rect as used at cub/code/SB_model48i/model.py:442.  The module is not vendored with the reference
    (SURVEY.md 8c): PARITY UNPINNED for this function; the convention restated here is the library's documented one
    (include/ups_b200.h): rows [cy - ph//2, cy - ph//2 + ph), columns [cx - pw//2, cx - pw//2 + pw), clipped."""
    N = centers.shape[0]
    out = torch.zeros(N, H, W)
    for n in range(N):
        cy, cx = int(centers[n, 0]), int(centers[n, 1])
        y0, x0 = cy - ph // 2, cx - pw // 2
        out[n, max(y0, 0):max(min(y0 + ph, H), 0), max(x0, 0):max(min(x0 + pw, W), 0)] = 1.0
    return out


def patch_masks(mask_hard, patch_size, gamma=3.0):
    """cub/code/SB_model48i/model.py:437-445 restated with the oracle's spatial softmax and moments."""
    from . import parts as P
    N, h, w, K = mask_hard.shape
    corrected = P.spatial_softmax(mask_hard * gamma)
    mu, _ = probs_to_mu_sigma(corrected, torch.ones(N, K))
    centers = (mu.reshape(N * K, 2) * h / 2.0 + h / 2.0).to(torch.int32)
    return draw_rect(centers, patch_size, patch_size, h, w).reshape(N, K, h, w).permute(0, 2, 3, 1).contiguous()
