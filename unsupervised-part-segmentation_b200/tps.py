"""Drop-in for `eddata.utils.tps` as the reference calls it (cub/code/SB_model48i/model.py:5,
300-309); the vendored source of that module is
baselines/unsupervised-disentangling/transformations.py:17-77,93-244."""
import math

import torch

from . import ops

_BASE = [[-0.5, -0.5], [0.5, -0.5], [-0.5, 0.5], [0.5, 0.5],
         [0.2, -0.2], [-0.2, 0.2], [0.2, 0.2], [-0.2, -0.2]]


class DotMap(dict):
    """attribute-access dict standing in for dotmap.DotMap (transformations.py:3,38)."""
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def draw_scalars(scal, tps_scal, rot_scal, off_scal, scal_var, rescal=1, augm_scal=None):
    """The ten scalars of the device draw (ups_tps_draw_solve, include/ups_b200.h) from tps_parameters' keyword
    arguments, in double: each range's lo and width hi - lo, rescal, and the rotation range as a fraction of a turn,
    rot_scal / (2 pi).  The C call rounds each to fp32 once.  rot_scal outside [0, pi] raises."""
    if augm_scal is not None:
        rescal = augm_scal
    if not 0.0 <= rot_scal <= math.pi:
        raise ValueError(f"rot_scal must lie in [0, pi], got {rot_scal}")
    vals = []
    for lo, hi in ((-0.2, 0.2), (-tps_scal, tps_scal), (-off_scal, off_scal),
                   (scal * (1.0 - scal_var), scal * (1.0 + scal_var))):
        vals += [float(lo), float(hi) - float(lo)]
    vals += [float(rescal), float(rot_scal) * (1.0 / (2.0 * math.pi))]
    return vals


def seed_args(seed):
    """seed (an int in [0, 2**64) or a one-element int64 CUDA tensor) -> the ops' (noise, seed, seed_value)."""
    if isinstance(seed, torch.Tensor):
        return ops.NOISE_DEVICE, seed, 0
    return ops.NOISE_INT, None, ops._seed_i64(seed)


def draw(seed, n_per_view, views, sample_offset, device, **tps_parameters):
    """ops.tps_draw for tps_parameters' keyword arguments: (coord, vector, offset, offset_2, t_scal, rot_mat, t_vector,
    T) of the rows [view 0 | view 1] (views = 2) or view 0 (views = 1), global samples sample_offset .. + n_per_view - 1."""
    scalars = draw_scalars(**tps_parameters)
    noise, st, value = seed_args(seed)
    if st is not None:
        device = st.device
    return ops.tps_draw(noise, st, value, int(sample_offset), int(n_per_view), int(views), scalars, torch.device(device))


def tps_parameters(batch_size, scal, tps_scal, rot_scal, off_scal, scal_var, rescal=1, augm_scal=None,
                   generator=None, device="cuda", seed=None, sample_offset=0, views=1):
    """transformations.py:17-39.  `augm_scal` is the kwarg the shipped config uses for `rescal`
    (cub/code/SB_model48i/train_cub_subset_tps.yaml:194).

    seed=None: ~50 random floats per sample, drawn on the host from `generator` (the reference draws them with
    tf.random_uniform) and moved to `device`.
    seed (an int in [0, 2**64), or a one-element int64 CUDA tensor that a captured CUDA graph reads at replay): the same
    fields drawn on the device, as a pure function of (seed, view, global sample) (csrc/canon_math.cuh, "the TPS
    parameters").  views=1: the rows are view 0 of samples sample_offset .. + batch_size - 1; views=2: batch_size is even
    and the rows are [view 0 | view 1] of samples sample_offset .. + batch_size / 2 - 1 (TrainModel.make_tps)."""
    if seed is not None:
        if generator is not None:
            raise ValueError("tps_parameters: pass a seed (device draw) or a generator (host draw), not both")
        if views not in (1, 2) or batch_size % views:
            raise ValueError(f"tps_parameters: views={views} needs a batch_size divisible by it, got {batch_size}")
        out = draw(seed, batch_size // views, views, sample_offset, device, scal=scal, tps_scal=tps_scal,
                   rot_scal=rot_scal, off_scal=off_scal, scal_var=scal_var, rescal=rescal, augm_scal=augm_scal)
        return DotMap(zip(("coord", "vector", "offset", "offset_2", "t_scal", "rot_mat"), out[:6]))
    if augm_scal is not None:
        rescal = augm_scal

    def U(shape, lo, hi):
        return torch.rand(shape, generator=generator, dtype=torch.float32) * (hi - lo) + lo

    coord = torch.tensor([_BASE], dtype=torch.float32).repeat(batch_size, 1, 1)
    coord = coord + U(coord.shape, -0.2, 0.2)
    vector = U(coord.shape, -tps_scal, tps_scal)
    offset = U((batch_size, 1, 2), -off_scal, off_scal)
    offset_2 = U((batch_size, 1, 2), -off_scal, off_scal)
    t_scal = U((batch_size, 2), scal * (1.0 - scal_var), scal * (1.0 + scal_var)) * rescal
    rot = U((batch_size, 1), -rot_scal, rot_scal)
    a, b = torch.cos(rot), torch.sin(rot)
    rot_mat = torch.stack([torch.cat([a, -b], 1), torch.cat([b, a], 1)], 1)
    d = dict(coord=coord, vector=vector, offset=offset, offset_2=offset_2, t_scal=t_scal, rot_mat=rot_mat)
    return DotMap({k: v.to(device, non_blocking=True) for k, v in d.items()})


def make_input_tps_param(tps_param, move_point=None, scal_point=None):
    """transformations.py:59-77 -> (coord, t_vector)."""
    coord = tps_param.coord
    t_vector = ops.tps_input_param(coord, tps_param.vector, tps_param.offset, tps_param.offset_2,
                                   tps_param.t_scal, tps_param.rot_mat)
    if move_point is not None and scal_point is not None:
        # crop branch (:70-72): two [B,8,2] broadcasts, outside the hot path -> plain torch
        coord = scal_point[:, None, :] * (coord + move_point)
        t_vector = scal_point[:, None, :] * t_vector
    else:
        assert move_point is None and scal_point is None
    return coord, t_vector


def ThinPlateSpline(U, coord, vector, out_size, n_c, move=None, scal=None):
    """transformations.py:93-244 -> (output [B,out,out,C], t_arr [B,out,out,2] = (y, x))."""
    assert U.dim() == 4 and U.shape[-1] == int(n_c), (list(U.shape), n_c)
    assert coord.shape == vector.shape and coord.shape[0] == U.shape[0] and tuple(coord.shape[1:]) == (8, 2), \
        list(coord.shape)
    assert (move is None) == (scal is None)
    # Gradients flow to the images U only.  The reference draws coord / vector / move / scal at random every step
    # (cub/code/SB_model48i/model.py:298-300): they are data, never variables.  A caller that asks for their gradient
    # gets an error here rather than a silently missing one (the TF graph would have propagated it).
    if any(t is not None and t.requires_grad for t in (coord, vector, move, scal)):
        raise ops.C.UpsError("ups_b200.ThinPlateSpline: coord / vector / move / scal must not require grad "
                             "(no gradient with respect to the warp parameters is implemented); detach them")
    T = ops.tps_solve(coord, vector)
    out, mesh = ops.tps_warp(U, coord, T, int(out_size), move, scal)
    return out, mesh
