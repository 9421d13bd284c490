"""Shared helpers for the parity tests: seeded synthetic inputs (SURVEY.md 8d) on the CPU,
identical tensors are fed to the oracle and (copied to cuda:0) to the kernels."""
import numpy as np
import torch

from oracle import tps as OT

RTOL, ATOL = 1e-4, 1e-5       # BASELINE.json north_star: fp32 within 1e-4 relative / 1e-5 absolute
CUB_TPS = dict(scal=0.8, tps_scal=0.15, rot_scal=0.2, off_scal=0.2, scal_var=0.1, augm_scal=1.0)
PENN_TPS = dict(scal=0.95, tps_scal=0.08, rot_scal=0.05, off_scal=0.2, scal_var=0.05, augm_scal=1.0)


def make_inputs(B, S, K, F, V=3, seed=0, tps=CUB_TPS, ties=False, tps_seed=1234):
    g = torch.Generator().manual_seed(seed)
    views = torch.rand(V, B, S, S, 3, generator=g) * 2 - 1
    l0 = torch.randn(B, S, S, K, generator=g)
    l1 = torch.randn(B, S, S, K, generator=g)
    if ties:  # exact ties and extreme logits in the first rows
        l0[:, 0] = torch.round(l0[:, 0])
        l1[:, 0] = torch.round(l1[:, 0])
        l0[:, 1] = l0[:, 1] * 40
        l1[:, 1, :, :] = 0.0
    feat = torch.randn(B, K, F, generator=g)
    gt = torch.Generator().manual_seed(tps_seed)
    prm = OT.tps_parameters(2 * B, generator=gt, **tps)
    coord, t_vector = OT.make_input_tps_param(prm)
    cot = dict(g_inj=torch.randn(B, S, S, F + K, generator=g), g_parts=torch.randn(K * B, S, S, 3, generator=g),
               g_pooled=torch.randn(B, K, 3, generator=g), g_m0=torch.randn(B, S, S, K, generator=g),
               g_m1=torch.randn(B, S, S, K, generator=g),
               g_warped=[torch.randn(B, S, S, 3, generator=g) for _ in range(V)])
    return dict(views=views, l0=l0, l1=l1, feat=feat, coord=coord, t_vector=t_vector, prm=prm, cot=cot)


def cuda(x):
    if isinstance(x, torch.Tensor):
        return x.cuda().contiguous()
    if isinstance(x, dict):
        return {k: cuda(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [cuda(v) for v in x]
    return x


def bits(t):
    return t.detach().cpu().contiguous().view(torch.int32)


def assert_bitexact(got, want, what=""):
    a, b = bits(got), bits(want)
    if not torch.equal(a, b):
        d = (got.detach().cpu().float() - want.float()).abs()
        n = (a != b).sum().item()
        raise AssertionError(f"{what}: {n}/{a.numel()} elements differ bitwise, max abs diff {d.max().item():.3e}")


def assert_close(got, want, what="", rtol=RTOL, atol=ATOL):
    g = got.detach().cpu().double()
    w = want.detach().double()
    assert g.shape == w.shape, (what, g.shape, w.shape)
    err = (g - w).abs()
    tol = atol + rtol * w.abs()
    if not bool((err <= tol).all()):
        i = torch.argmax(err - tol)
        raise AssertionError(f"{what}: {(err > tol).sum().item()}/{err.numel()} outside rtol={rtol} atol={atol}; "
                             f"worst |d|={err.flatten()[i].item():.3e} at ref={w.flatten()[i].item():.6e}")


def own_error_atol(want32, want64, atol=ATOL):
    """Absolute tolerance for a quantity that is a long fp32 sum (dfeat, pooled, weight gradients): the north-star
    1e-5 plus twice the distance of the fp32 ORACLE from the float64 value of the same expression.  Two valid fp32
    summation orders (the oracle's and the kernel's) each sit that far from the exact value; entries that cancel to ~0
    cannot agree more closely than that, whatever the kernel does.  Measured per test, not assumed (VERDICT r1 weak #1)."""
    return atol + 2.0 * float((want32.detach().double().cpu() - want64.detach().double().cpu()).abs().max())


def check_tps_against_fixture(out, mesh, ref_out, ref_mesh, S, strict, what=""):
    """Warped image and sample mesh against a reference-generated TPS fixture (tests/golden/tps_*.npz).

    strict (the shipped CUB / PennAction parameter ranges): EVERY pixel within the north-star 1e-4 rel / 1e-5 abs, and
    no pixel whose bilinear cell differs from the reference's (floor-boundary whitelist must be empty).
    not strict (the 4x exaggerated `big` warp, and the identity warp whose samples sit exactly ON cell borders): pixels
    whose cell differs are counted and excluded (returned), the others may add the bound that the measured
    sample-position difference implies: |d out| <= max|U[x+1] - U[x]| * (|dX| + |dY|) <= 2 * (|dX| + |dY|) for U in [-1, 1].
    Returns (n_whitelisted, max_abs_mesh_diff)."""
    out, mesh = out.detach().cpu().double(), mesh.detach().cpu().double()
    ref_out, ref_mesh = ref_out.double(), ref_mesh.double()
    dpix = (mesh - ref_mesh).abs() * S / 2
    same = (torch.floor((mesh + 1) * S / 2) == torch.floor((ref_mesh + 1) * S / 2)).all(-1)
    n_white = int((~same).sum())
    tol = ATOL + RTOL * ref_out.abs()
    if strict:
        assert n_white == 0, f"{what}: {n_white} pixels sample a different bilinear cell than the reference"
    else:
        tol = tol + 2.0 * dpix.sum(-1, keepdim=True)
    err = (out - ref_out).abs()
    bad = (err > tol).any(-1) & same
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{same.numel()} pixels outside tolerance, "
                                 f"worst {float(err[same].max()):.3e}, mesh diff {float((mesh - ref_mesh).abs().max()):.3e}")
    return n_white, float((mesh - ref_mesh).abs().max())
