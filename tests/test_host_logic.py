"""CPU tier: host-side logic added in round 2 — the path configuration mirror, the stream handle that carries its
device, the stand-in modules' oracle (float64 gradcheck), the fp64 reduction references, and the bucket / default
tables of the data-parallel wrapper.  No GPU work."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def ups():
    import __graft_entry__ as ge
    ge.build()
    import ups_b200
    return ups_b200


def test_path_config_mirrors_the_reference_keys(ups):
    from util import CUB_TPS, PENN_TPS
    from ups_b200 import configs
    assert configs.CUB_TPS == CUB_TPS and configs.PENN_TPS == PENN_TPS          # tests keep their own copy of the constants
    ship = configs.CUB_SHIPPED
    # cub/code/SB_model48i/train_cub_subset_tps.yaml:19-20,132,139
    assert (ship.batch_size, ship.spatial_size, ship.n_parts, ship.local_app_size) == (8, 128, 25, 64)
    cfg = configs.PathConfig.from_dict(dict(batch_size=4, n_parts=16, use_tps=False, lr=1e-4, model="x"))
    assert cfg.batch_size == 4 and cfg.n_parts == 16 and cfg.use_tps is False and "lr" not in cfg.to_dict()
    assert set(cfg.tps_parameters) == {"scal", "tps_scal", "rot_scal", "off_scal", "scal_var", "augm_scal"}
    assert configs.PENNACTION_BENCH.batch_size == 512 and configs.DEEPFASHION_BENCH.spatial_size == 256


def test_stream_handle_is_an_int_with_a_device(ups):
    C = ups._cabi
    h = C.StreamHandle(1234, 3)
    assert int(h) == 1234 and h.device_index == 3
    assert ctypes.c_void_p.from_param(h) is not None          # ctypes takes it where a void* is expected


def test_standin_oracle_gradients_are_the_analytic_ones():
    from oracle import standin as S
    g = torch.Generator().manual_seed(0)
    B, K, F, P = 2, 5, 4, 12
    pooled, dfeat = torch.randn(B, K, 3, generator=g), torch.randn(B, K, F, generator=g)
    Wlin, blin = torch.randn(3, F, generator=g), torch.randn(F, generator=g)
    t = S.tail_grads(pooled, dfeat, Wlin, blin)
    want = torch.cat([(pooled.reshape(-1, 3).t().double() @ dfeat.reshape(-1, F).double()).reshape(-1), dfeat.double().sum((0, 1))])
    assert torch.allclose(t, want, atol=1e-12)
    labels = torch.randint(0, K, (B, P), generator=g)
    feat, g_recon = torch.randn(B, K, F, generator=g), torch.randn(B, P, 3, generator=g)
    Whead, bhead = torch.randn(F + K, 3, generator=g), torch.randn(3, generator=g)
    h = S.head_grads(g_recon, labels, feat, Whead, bhead)
    R = torch.zeros(B, K, 3, dtype=torch.float64)
    for b in range(B):
        for p in range(P):
            R[b, labels[b, p]] += g_recon[b, p].double()
    dW = torch.cat([torch.einsum("bkf,bkc->fc", feat.double(), R), R.sum(0)], 0)
    assert torch.allclose(h, torch.cat([dW.reshape(-1), R.sum((0, 1))]), atol=1e-12)
    # forward: recon of a pixel = Whead rows of its part's features + the one-hot row + bias
    rec = S.head_fwd(labels, feat, Whead, bhead)
    k = int(labels[1, 3])
    assert torch.allclose(rec[1, 3], feat[1, k] @ Whead[:F] + Whead[F + k] + bhead, atol=1e-5)


def test_fp64_reduction_references_agree_with_the_fp32_oracle():
    """oracle/step.py::reduction_refs_fp64 evaluates the same sums as autograd of the fp32 oracle (to fp32 rounding)."""
    from oracle import step as OS
    from util import make_inputs
    B, S, K, F, V = 2, 16, 8, 16, 3
    inp = make_inputs(B, S, K, F, V, seed=3)
    cot = dict(inp["cot"])
    out, grad = OS.step_forward_backward([v for v in inp["views"]], inp["coord"], inp["t_vector"], inp["l0"], inp["l1"],
                                         inp["feat"], cot, views_grad=True)
    r64 = OS.reduction_refs_fp64([v for v in inp["views"]], inp["coord"], inp["t_vector"], out, cot, views_grad=True)
    assert torch.allclose(r64["pooled"].float(), out["pooled"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(r64["dfeat"].float(), grad["dfeat"], rtol=1e-5, atol=1e-5)
    for a, b in zip(r64["dviews"], grad["dviews"]):
        assert torch.allclose(a.float(), b, rtol=1e-5, atol=1e-5)


def test_dp_tables(ups):
    from ups_b200 import dp
    assert dp.default_main_bucket(8) == "before_k4" and dp.default_main_bucket(4) == "after_k4" == dp.default_main_bucket(2)
    assert dp.default_allreduce_ctas(8) == 16 and dp.default_allreduce_ctas(4) == 64 and dp.default_allreduce_ctas(2) == 128
    b = dp.two_buckets(33_300_000)
    assert b[1][1] == dp.TAIL_BUCKET_FLOATS >= 4 * 64 + (64 + 32) * 3 + 3 + 3      # both stand-in gradients fit (K <= 32, F = 64)
    # the gloo reducer handles sub-range launches (part = (i, n)) on CPU tensors without a process group (world 1: no-op)
    red = dp.GradAllReducer(flat_grads=torch.ones(64), world_size=1)
    red.launch(0, part=(1, 2))
    assert float(red.flat.sum()) == 64.0


def test_bench_knows_the_bytes_of_every_call_of_the_fused_step(ups):
    """bench.py's roofline is keyed by C-ABI call name: every `ups_step_*` / `ups_tps_warp_*` call that step.py issues
    (whatever its argument form: plain, `_planes`, `_rows`) must have algorithmic bytes, and the ones with a committed
    ncu capture must find their kernel in profiles/ncu_traffic.json.  (A renamed entry point once left `roofline.frac`
    null.)"""
    import importlib.util
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    src = open(os.path.join(root, "unsupervised-part-segmentation_b200", "step.py")).read()
    names = set(re.findall(r'"(ups_step_[a-z0-9_]+|ups_tps_warp_[a-z0-9_]+)"', src))
    assert {"ups_step_warp_decode_fwd_rows", "ups_step_encode_fwd_rows", "ups_step_decode_bwd_tc_rows",
            "ups_step_encode_bwd_rows"} <= names
    for n in names:
        assert bench.call_bytes(n, 16, 64, 3, 256, 16384), n
    assert bench.base_call("ups_step_encode_fwd_planes") == "ups_step_encode_fwd"
    for n in ("ups_step_warp_decode_fwd_rows", "ups_step_encode_fwd_rows", "ups_step_decode_bwd_tc_rows", "ups_step_encode_bwd_rows"):
        traffic, source = bench.ncu_traffic(n, "cub", 256)
        assert traffic and traffic > 0.9 * bench.call_bytes(n, 16, 64, 3, 256, 16384) * 0.5 and source, n


def test_bench_dump_outputs_fits_64_mb_and_samples_the_same_entries(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole, integer ones as float64; arrays too large for 64 MB in
    all are written as a 1-D sample taken at the same positions on every call, so two runs compare entry for entry."""
    import importlib.util
    import os

    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    base = torch.arange(16_000_000, dtype=torch.float32)          # 64 MB: each entry holds its own flat position
    out = {f"big{i}": base for i in range(12)}
    out.update(small=torch.randn(4, 5, generator=g), labels=torch.randint(0, 16, (2, 8, 8), generator=g), absent=None)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted([f"big{i}.npy" for i in range(12)] + ["labels.npy", "small.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    load = lambda d, n: np.load(tmp_path / d / f"{n}.npy")  # noqa: E731
    assert load("a", "small").dtype == np.float32 and np.array_equal(load("a", "small"), out["small"].numpy())
    assert load("a", "labels").dtype == np.float64 and np.array_equal(load("a", "labels"), out["labels"].numpy())
    s = load("a", "big0")
    assert s.dtype == np.float32 and s.ndim == 1 and 0 < s.size < base.numel()
    assert np.all(np.diff(s) > 0) and s[-1] < base.numel()                  # distinct positions, in order
    assert np.array_equal(s, load("b", "big0")) and np.array_equal(s, load("a", "big11"))
