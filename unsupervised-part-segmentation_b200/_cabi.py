"""ctypes binding of libups_b200.so (include/ups_b200.h).  No fallback: if the library is
missing or a call fails, this raises."""
import ctypes
import os

from . import build as _build

c_f = ctypes.c_void_p      # device pointers travel as integers
c_i = ctypes.c_int
c_ll = ctypes.c_longlong
c_sz = ctypes.c_size_t
c_fl = ctypes.c_float
c_u64 = ctypes.c_ulonglong

_SIGS = {
    "ups_views_u8_to_f32": [c_f, c_f, c_ll, c_f],
    "ups_labels_i64_to_u8": [c_f, c_f, c_ll, c_f],
    "ups_tps_input_param": [c_f] * 7 + [c_i, c_f],
    "ups_tps_solve": [c_f, c_f, c_f, c_i, c_f],
    "ups_tps_warp_fwd": [c_f] * 7 + [c_i] * 6 + [c_f],
    "ups_tps_warp_bwd": [c_f] * 6 + [c_i] * 6 + [c_f],
    "ups_tps_warp_pair_fwd": [c_f] * 6 + [c_i] * 7 + [c_f],
    "ups_tps_warp_pair_bwd": [c_f] * 6 + [c_i] * 7 + [c_f],
    "ups_part_softmax_fwd": [c_f, c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_part_softmax_bwd": [c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_part_softmax_bwd2": [c_f, c_f, c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_axpy": [c_f, c_f, c_ll, c_fl, c_f],
    "ups_views_cotangent": [c_f, c_f, c_f, c_i, c_i, c_ll, c_f],
    "ups_spatial_softmax_fwd": [c_f, c_f, c_i, c_i, c_i, c_f],
    "ups_spatial_softmax_bwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_f],
    "ups_hard_max_fwd": [c_f, c_f, c_ll, c_i, c_f],
    "ups_straight_through_fwd": [c_f, c_f, c_f, c_ll, c_f],
    "ups_argmax_fwd": [c_f, c_f, c_ll, c_i, c_f],
    "ups_one_hot_fwd": [c_f, c_f, c_ll, c_i, c_f],
    "ups_mask_parts_fwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_i, c_i, c_f],
    "ups_mask_parts_bwd": [c_f] * 5 + [c_i] * 5 + [c_f],
    "ups_partwise_fold": [c_f, c_f, c_i, c_i, c_i, c_i, c_f],
    "ups_partwise_unfold": [c_f, c_f, c_i, c_i, c_i, c_i, c_f],
    "ups_part_pool_fwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_i, c_i, c_fl, c_f, c_sz, c_f],
    "ups_part_pool_bwd": [c_f] * 5 + [c_i] * 5 + [c_fl, c_f],
    "ups_part_unpool_fwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_i, c_f],
    "ups_part_unpool_bwd": [c_f] * 5 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_part_inject_fwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_i, c_f],
    "ups_part_inject_bwd": [c_f] * 5 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_part_gather_fwd": [c_f, c_f, c_f, c_i, c_i, c_i, c_i, c_f],
    "ups_step_encode_fwd": [c_f] * 5 + [c_i] * 3 + [c_f, c_sz, c_f],
    "ups_step_decode_fwd": [c_f] * 5 + [c_i] * 4 + [c_f],
    "ups_step_decode_bwd": [c_f] * 6 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_decode_bwd_tc": [c_f] * 6 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_encode_bwd": [c_f] * 7 + [c_i] * 3 + [c_f],
    "ups_mask_moments_fwd": [c_f] * 5 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_mask_moments_bwd": [c_f] * 5 + [c_i] * 4 + [c_f],
    "ups_categorical_kl_fwd": [c_f, c_f, c_ll, c_i, c_f, c_sz, c_f],
    "ups_categorical_kl_bwd": [c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_mumford_shah_fwd": [c_f, c_fl, c_fl] + [c_f] * 5 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_mumford_shah_bwd": [c_f, c_fl, c_fl] + [c_f] * 5 + [c_i] * 4 + [c_f],
    "ups_logit_priors_fwd": [c_f, c_f] + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_logit_priors_bwd": [c_f, c_f, c_f] + [c_i] * 4 + [c_f],
    "ups_mean_field_sample_fwd": [c_f, c_f, c_fl, c_f, c_ll, c_f],
    "ups_part_softmax_sampled_fwd": [c_f, c_f, c_fl, c_f, c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_weak_xent_fwd": [c_f, c_i, c_f, c_ll, c_i, c_f, c_sz, c_f],
    "ups_weak_xent_bwd": [c_f, c_i, c_f, c_f, c_ll, c_i, c_f],
    "ups_mask2rgb_fwd": [c_f, c_f, c_i, c_f, c_ll, c_i, c_f],
    "ups_inject_conv_table_fwd": [c_f, c_f, c_f] + [c_i] * 4 + [c_f],
    "ups_inject_conv_table_bwd": [c_f] * 5 + [c_i] * 4 + [c_f],
    "ups_inject_conv_fwd": [c_f] * 4 + [c_i] * 5 + [c_f],
    "ups_parts_conv_fwd": [c_f] * 5 + [c_i] * 6 + [c_f],
    "ups_parts_conv_bwd": [c_f] * 9 + [c_i] * 6 + [c_f, c_sz, c_f],
    "ups_inject_conv_bwd_plan": [c_i] * 5 + [c_f],
    "ups_inject_conv_bwd": [c_f] * 8 + [c_i] * 5 + [c_f, c_sz, c_f],
    "ups_copy_rows": [c_f, c_ll, c_f, c_ll, c_ll, c_i, c_i, c_fl, c_f],
    "ups_step_encode_fwd_planes": [c_f] * 5 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_encode_bwd_planes": [c_f] * 7 + [c_i] * 4 + [c_f],
    "ups_tps_warp_bwd_sum": [c_f, c_f, c_f, c_i, c_i, c_f, c_f, c_f, c_f] + [c_i] * 7 + [c_f],
    "ups_step_decode_fwd_rows": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_f],
    "ups_step_encode_fwd_rows": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_decode_bwd_rows": [c_f, c_f, c_f, c_i, c_f, c_f, c_f] + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_decode_bwd_tc_rows": [c_f, c_f, c_f, c_i, c_f, c_f, c_f] + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_step_encode_bwd_rows": [c_f] * 5 + [c_i] + [c_f] * 2 + [c_i] * 4 + [c_f],
    "ups_step_warp_decode_fwd_rows": [c_f] * 6 + [c_i] * 3 + [c_f, c_i] + [c_f] * 4 + [c_i] * 3 + [c_f],
    "ups_draw_rect_fwd": [c_f, c_f] + [c_i] * 5 + [c_f],
    "ups_step_warp_decode_fwd": [c_f] * 6 + [c_i] * 3 + [c_f] * 5 + [c_i] * 3 + [c_f],
    "ups_dp_allreduce": [c_f, c_f, c_f, c_i, c_i, c_ll, c_fl, c_i, c_f],
    "ups_standin_tail_fwd": [c_f] * 4 + [c_i] * 4 + [c_f],
    "ups_standin_tail_bwd": [c_f] * 3 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_standin_head_fwd": [c_f] * 5 + [c_i] * 4 + [c_f],
    "ups_standin_head_bwd": [c_f] * 4 + [c_i] * 4 + [c_f, c_sz, c_f],
    "ups_normal_philox_fwd": [c_u64, c_i, c_ll, c_ll, c_i, c_f, c_f],
    "ups_part_softmax_sampled_philox_fwd": [c_f, c_u64, c_i, c_ll, c_fl, c_f, c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_step_decode_fwd_noise": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_u64, c_ll, c_fl, c_f],
    "ups_step_encode_fwd_noise": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_f, c_sz] + [c_u64, c_ll, c_fl, c_f],
    "ups_step_warp_decode_fwd_noise": [c_f] * 6 + [c_i] * 3 + [c_f, c_i] + [c_f] * 4 + [c_i] * 3 + [c_u64, c_ll, c_fl, c_f],
    "ups_normal_philox_fwd_dseed": [c_f, c_i, c_ll, c_ll, c_i, c_f, c_f],
    "ups_part_softmax_sampled_philox_fwd_dseed": [c_f, c_f, c_i, c_ll, c_fl, c_f, c_f, c_f, c_f, c_ll, c_i, c_f],
    "ups_step_decode_fwd_noise_dseed": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_f, c_ll, c_fl, c_f],
    "ups_step_encode_fwd_noise_dseed": [c_f, c_i] + [c_f] * 4 + [c_i] * 4 + [c_f, c_sz] + [c_f, c_ll, c_fl, c_f],
    "ups_tps_draw_solve": [c_u64, c_ll, c_i, c_i] + [c_fl] * 10 + [c_f] * 9,
    "ups_tps_draw_solve_dseed": [c_f, c_ll, c_i, c_i] + [c_fl] * 10 + [c_f] * 9,
}

OP_TPS_SOLVE, OP_POOL, OP_INJECT_BWD, OP_POOL_BWD, OP_STEP, OP_MOMENTS, OP_KL = 0, 1, 2, 3, 4, 5, 6
OP_MUMFORD_SHAH, OP_LOGIT_PRIORS, OP_WEAK_XENT = 7, 8, 9


class UpsError(RuntimeError):
    pass


def _load():
    path = os.environ.get("UPS_B200_LIB", _build.LIB)
    if not os.path.exists(path):
        raise UpsError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(path)
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = c_i
    lib.ups_version.restype = ctypes.c_char_p
    lib.ups_last_error_string.restype = ctypes.c_char_p
    lib.ups_launch_count.restype = c_ll
    lib.ups_launch_count_reset.restype = None
    lib.ups_workspace_bytes.argtypes = [c_i] * 5
    lib.ups_workspace_bytes.restype = c_sz
    lib.ups_inject_conv_workspace_bytes.argtypes = [c_i] * 5
    lib.ups_inject_conv_workspace_bytes.restype = c_sz
    lib.ups_parts_conv_bwd_workspace_bytes.argtypes = [c_i] * 5
    lib.ups_parts_conv_bwd_workspace_bytes.restype = c_sz
    lib.ups_standin_workspace_bytes.argtypes = [c_i] * 4
    lib.ups_standin_workspace_bytes.restype = c_sz
    lib.ups_dp_allreduce_signal_bytes.argtypes = [c_i] * 2
    lib.ups_dp_allreduce_signal_bytes.restype = c_sz
    return lib, path


lib, LIB_PATH = _load()


class StreamHandle(int):
    """A cudaStream_t (as an integer) that remembers the index of the device it belongs to."""

    def __new__(cls, stream, device_index):
        self = super().__new__(cls, stream)
        self.device_index = device_index
        return self


def call(name, *args):
    """Invoke one C-ABI entry point.  The stream is the last argument of every entry point; when it is a
    StreamHandle of a device other than the calling thread's current one, that device is made current for
    the call (the library launches on the current device and never calls cudaSetDevice itself)."""
    st = args[-1] if args else None
    if isinstance(st, StreamHandle) and st.device_index is not None:
        import torch
        if torch.cuda.current_device() != st.device_index:
            with torch.cuda.device(st.device_index):
                rc = getattr(lib, name)(*args)
        else:
            rc = getattr(lib, name)(*args)
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        raise UpsError(f"{name} -> {rc}: {lib.ups_last_error_string().decode()}")


def version():
    return lib.ups_version().decode()


def launch_count():
    return int(lib.ups_launch_count())


def launch_count_reset():
    lib.ups_launch_count_reset()


def inject_conv_workspace_bytes(B, H, W, K, Co):
    return int(lib.ups_inject_conv_workspace_bytes(B, H, W, K, Co))


def inject_conv_bwd_plan(B, H, W, K, Co):
    out = (ctypes.c_int * 6)()
    call("ups_inject_conv_bwd_plan", B, H, W, K, Co, ctypes.cast(out, ctypes.c_void_p))
    return dict(zip(("variant", "tile_rows", "ctas_per_sample", "tiles_per_cta", "smem_bytes", "tiles"), list(out)))


def parts_conv_bwd_workspace_bytes(B, H, W, K, Co):
    return int(lib.ups_parts_conv_bwd_workspace_bytes(B, H, W, K, Co))


def workspace_bytes(op, B, P, K, F):
    return int(lib.ups_workspace_bytes(op, B, P, K, F))
