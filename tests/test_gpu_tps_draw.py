"""-m gpu: the TPS parameters drawn on the device from a seed (ups_tps_draw_solve, ups::tps_draw, make_tps(seed=...),
PartStep.forward(tps_seed=...)).

  a. the device draw equals the host build of the same header bit for bit, with an int and with a device seed;
  b. coord / t_vector / T of the fused launch equal ups_tps_input_param + ups_tps_solve on its raw fields;
  c. make_tps(seed=...) equals ThinPlateSpline on the regenerated parameters, and the oracle on a slice;
  d. PartStep(tps_seed=...) equals PartStep fed the drawn coord / t_vector, with the same C-ABI launches;
  e. one step of 2n samples equals two steps of n at sample offsets 0 and n;
  f. a model-order training step with make_tps inside is captured in one CUDA graph that redraws at every replay;
  g. opcheck and torch.compile(fullgraph=True); h. errors."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import tps as OT
from oracle import tps_draw as OD
from util import CUB_TPS, PENN_TPS, assert_close, cuda, make_inputs
from test_gpu_model_order import LEVEL, Tiny, _views, assert_bitexact

pytestmark = pytest.mark.gpu

SEED = 0x0DD5_EED0_1234_5678
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "unsupervised-part-segmentation_b200",
                    "csrc")
RAW = ("coord", "vector", "offset", "offset_2", "t_scal", "rot_mat")


@pytest.fixture(scope="module")
def ups():
    import ups_b200
    return ups_b200


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("canon_host") / "libups_canon_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(CSRC, "canon_host.cpp"),
                           "-o", so])
    return ctypes.CDLL(so)


def _seed_tensor(seed):
    from ups_b200 import ops
    return torch.tensor([ops._seed_i64(seed)], dtype=torch.int64, device="cuda")


def host_rows(host, seed, n_per_view, views, sample_offset, kw):
    """The rows [view 0 | view 1] from the host build (canon_host.cpp::ups_host_tps_draw)."""
    s = np.ascontiguousarray(OD.draw_scalars(**kw), np.float32)
    per = []
    for v in range(views):
        o = dict(coord=np.empty((n_per_view, 8, 2), np.float32), vector=np.empty((n_per_view, 8, 2), np.float32),
                 offset=np.empty((n_per_view, 1, 2), np.float32), offset_2=np.empty((n_per_view, 1, 2), np.float32),
                 t_scal=np.empty((n_per_view, 2), np.float32), rot_mat=np.empty((n_per_view, 2, 2), np.float32))
        host.ups_host_tps_draw(ctypes.c_ulonglong(seed), ctypes.c_int(v), ctypes.c_ulonglong(sample_offset),
                               ctypes.c_longlong(n_per_view), s.ctypes.data_as(ctypes.c_void_p),
                               *[o[k].ctypes.data_as(ctypes.c_void_p) for k in RAW])
        per.append(o)
    return {k: torch.from_numpy(np.concatenate([p[k] for p in per])) for k in RAW}


def device_rows(ups, seed, n_per_view, views, sample_offset, kw):
    return ups.tps.draw(seed, n_per_view, views, sample_offset, "cuda", **kw)


# ---------------------------------------------------------------- a. the device draw is the host build's
DRAWS = [pytest.param(CUB_TPS, 256, 1000, id="cub_2x256"), pytest.param(PENN_TPS, 512, 3 * 512, id="penn_2x512")]


@pytest.mark.parametrize("kw,n,offset", DRAWS)
def test_device_draw_equals_host(ups, host, kw, n, offset):
    want = host_rows(host, SEED, n, 2, offset, kw)
    by_value = device_rows(ups, SEED, n, 2, offset, kw)
    seed_t = _seed_tensor(SEED)
    by_address = device_rows(ups, seed_t, n, 2, offset, kw)
    for i, k in enumerate(RAW):
        assert_bitexact(by_value[i], want[k].cuda(), f"int seed: {k}")
        assert_bitexact(by_address[i], want[k].cuda(), f"device seed: {k}")
    for i in (6, 7):
        assert_bitexact(by_address[i], by_value[i], "t_vector / T")
    seed_t.fill_(ups.ops._seed_i64(SEED + 1))
    again = device_rows(ups, seed_t, n, 2, offset, kw)
    assert not torch.equal(again[0], by_address[0]), "a new value in the seed tensor must give a new draw"
    assert_bitexact(again[0], host_rows(host, SEED + 1, n, 2, offset, kw)["coord"].cuda(), "coord, second seed")


# ---------------------------------------------------------------- b. the fused launch is input_param + solve
@pytest.mark.parametrize("kw,n,offset", DRAWS)
def test_fused_equals_input_param_and_solve(ups, kw, n, offset):
    coord, vector, off, off2, ts, rot, tv, T = device_rows(ups, 2 ** 64 - 3, n, 2, offset, kw)
    tv_want = ups.ops.tps_input_param(coord, vector, off, off2, ts, rot)
    assert_bitexact(tv, tv_want, "t_vector")
    assert_bitexact(T, ups.ops.tps_solve(coord, tv_want), "T")


# ---------------------------------------------------------------- c. make_tps(seed=...)
@pytest.mark.parametrize("V", [3, 2])
def test_make_tps_seed_equals_thin_plate_spline(ups, V):
    B, S, offset = 256, 128, 4096
    views = _views(B, S, 3)[:V]
    for seed in (SEED, _seed_tensor(SEED)):
        got = ups.make_tps(views, CUB_TPS, seed=seed, sample_offset=offset)
        prm = ups.tps.tps_parameters(2 * B, seed=SEED, sample_offset=offset, views=2, **CUB_TPS)
        coord, tv = ups.make_input_tps_param(prm)
        want, _ = ups.ThinPlateSpline(torch.cat(views[:2]), coord, tv, S, 3)
        assert len(got) == V
        assert_bitexact(got[0], want[:B], "view 0")
        assert_bitexact(got[1], want[B:], "view 1")
        if V > 2:
            want_t, _ = ups.ThinPlateSpline(views[2], coord[:B], tv[:B], S, 3)   # the target uses view 0's rows
            assert_bitexact(got[2], want_t, "target view")


def test_make_tps_seed_matches_the_oracle(ups):
    """A B = 8 CUB slice against oracle.tps.make_tps_given on the drawn parameters (the bar of test_gpu_tps.py)."""
    B, S = 8, 128
    views = [v.cpu() for v in _views(B, S, 5)]
    got = ups.make_tps([v.cuda() for v in views], CUB_TPS, seed=SEED, sample_offset=77)
    prm = OD.tps_parameters(SEED, B, 2, 77, **CUB_TPS)
    coord, tv = OT.make_input_tps_param(prm)
    for a, b in zip(got, OT.make_tps_given(views, coord, tv)):
        assert_bitexact(a, b.cuda(), "make_tps view")


# ---------------------------------------------------------------- d. PartStep(tps_seed=...)
# (name, B, S, K, F, V, views_grad, UPS_FUSE_FWD)
STEPS = [
    ("fused_k1k3", 256, 128, 16, 64, 3, False, "1"),
    ("two_launch", 16, 64, 16, 64, 3, False, "0"),
    ("padded_k25", 16, 64, 25, 64, 3, False, "1"),
    ("views_grad", 16, 64, 16, 64, 3, True, "1"),
    ("two_views", 16, 64, 8, 32, 2, False, "1"),
]


def _record(monkeypatch):
    from ups_b200 import _cabi as C
    calls, real = [], C.call
    monkeypatch.setattr(C, "call", lambda name, *a: (calls.append(name), real(name, *a))[1])
    return calls


@pytest.mark.parametrize("case", STEPS, ids=[c[0] for c in STEPS])
@pytest.mark.parametrize("seed_kind", ["int", "device"])
def test_partstep_seed_equals_given_coord(ups, monkeypatch, case, seed_kind):
    from ups_b200 import _cabi as C
    from ups_b200.step import PartStep
    name, B, S, K, F, V, vg, fuse = case
    monkeypatch.setenv("UPS_FUSE_FWD", fuse)
    inp = cuda(make_inputs(B, S, K, F, V=V, seed=9))
    cot = inp["cot"]
    g_warped = torch.stack(cot["g_warped"]) if vg else None
    seed = SEED if seed_kind == "int" else _seed_tensor(SEED)
    steps = [PartStep(B, S, K, F, n_views=V, views_grad=vg, sample_offset=3 * B) for _ in range(2)]
    assert steps[0].fuse_fwd == (fuse == "1")
    runs = []
    for i, st in enumerate(steps):
        calls = _record(monkeypatch)
        C.launch_count_reset()
        if i == 0:
            out = st.forward(inp["views"], None, None, inp["l0"], inp["l1"], inp["feat"], tps_seed=seed)
            drawn = {k: v.clone() for k, v in st.tps_drawn().items()}
        else:
            out = st.forward(inp["views"], drawn["coord"], drawn["t_vector"], inp["l0"], inp["l1"], inp["feat"])
        grad = st.backward(cot["g_inj"], cot["g_parts"], cot["g_pooled"], cot["g_m0"], cot["g_m1"], g_warped)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in out.items() if v is not None},
                     {k: v.clone() for k, v in grad.items()}, list(calls), C.launch_count()))
        monkeypatch.undo()
        monkeypatch.setenv("UPS_FUSE_FWD", fuse)
    (o_s, g_s, calls_s, n_s), (o_g, g_g, calls_g, n_g) = runs
    for k in o_g:
        if o_g[k].dtype == torch.float32:
            assert_bitexact(o_s[k], o_g[k], f"{name}: {k}")
        else:
            assert torch.equal(o_s[k], o_g[k]), k
    for k in g_g:
        if k == "dviews":          # a scatter-add of atomics: the order of the sums differs between runs
            assert_close(g_s[k], g_g[k].cpu(), k, rtol=1e-3, atol=1e-3)
        else:
            assert_bitexact(g_s[k], g_g[k], f"{name}: {k}")
    assert n_s == n_g, (n_s, n_g)
    solve = "ups_tps_draw_solve_dseed" if seed_kind == "device" else "ups_tps_draw_solve"
    assert calls_s == [solve if c == "ups_tps_solve" else c for c in calls_g]


def test_partstep_argument_errors(ups):
    from ups_b200.step import PartStep
    B, S, K, F = 2, 32, 16, 32
    d = cuda(make_inputs(B, S, K, F, V=3, seed=1))
    st = PartStep(B, S, K, F, n_views=3)
    with pytest.raises(ValueError, match="not both"):
        st.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"], tps_seed=1)
    with pytest.raises(ValueError, match="coord and t_vector, or tps_seed"):
        st.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"])


# ---------------------------------------------------------------- e. the batch split
def test_partstep_split_equals_whole(ups):
    """What DataParallelPartStep relies on: a step of 2n samples warps what two steps of n at sample offsets 0 and n
    warp (row v * B + b is view v of global sample sample_offset + b)."""
    from ups_b200.step import PartStep
    n, S, K, F = 32, 64, 16, 64
    d = cuda(make_inputs(2 * n, S, K, F, V=3, seed=4))
    whole = PartStep(2 * n, S, K, F, n_views=3)
    ow = whole.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"], tps_seed=SEED)
    cw = whole.tps_drawn()["coord"].view(2, 2 * n, 8, 2)
    for h in range(2):
        part = PartStep(n, S, K, F, n_views=3, sample_offset=h * n)
        sl = slice(h * n, (h + 1) * n)
        op = part.forward(d["views"][:, sl].contiguous(), None, None, d["l0"][sl].contiguous(), d["l1"][sl].contiguous(),
                          d["feat"][sl].contiguous(), tps_seed=SEED)
        assert_bitexact(op["warped"], ow["warped"][:, sl], f"half {h}: warped")
        assert_bitexact(part.tps_drawn()["coord"].view(2, n, 8, 2), cw[:, sl], f"half {h}: coord")
        assert_bitexact(op["m1"], ow["m1"][sl], f"half {h}: m1")


# ---------------------------------------------------------------- f. one CUDA graph with make_tps inside
def _train_step(ups, model, raw_views, seed, taps):
    warped = ups.make_tps(raw_views, CUB_TPS, seed=seed)
    loss, out = model(warped, True, seed, LEVEL, taps)
    loss.backward()
    return {**{k: out[k] for k in ("m0", "m1", "labels0")}, "warped1": warped[1], "warped2": warped[2], **taps}


@pytest.mark.parametrize("K", [25, 16])
def test_cuda_graph_redraws_the_warp_per_replay(ups, deterministic, K):
    B, S, F = 2, 64, 32
    raw = _views(B, S, 16)
    model = Tiny(K, F, seed=3).cuda()
    seed_t = _seed_tensor(0)

    def run():
        taps = {}
        return _train_step(ups, model, raw, seed_t, taps)

    def eager(value):
        model.zero_grad(set_to_none=True)
        seed_t.fill_(ups.ops._seed_i64(value))
        r = {k: v.clone() for k, v in run().items()}
        torch.cuda.synchronize()
        return r

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            model.zero_grad(set_to_none=True)
            run()
    torch.cuda.current_stream().wait_stream(side)
    model.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    static = {}
    with torch.cuda.graph(graph):
        static.update(run())
    values = (3, SEED, 2 ** 64 - 5)
    results = []
    for value in values:
        seed_t.fill_(ups.ops._seed_i64(value))
        graph.replay()
        torch.cuda.synchronize()
        results.append({k: v.clone() for k, v in static.items()})
    for value, got in zip(values, results):
        want = eager(value)
        for k in ("warped1", "warped2", "m0", "m1", "labels0", "dl0", "dl1", "dfeat"):
            if want[k].dtype == torch.float32:
                assert_bitexact(got[k], want[k], f"seed={value}: {k}")
            else:
                assert torch.equal(got[k], want[k]), (value, k)
    assert not torch.equal(results[0]["warped1"], results[1]["warped1"]), "replays with different seeds must warp differently"


@pytest.fixture
def deterministic():
    prev = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev


def test_int_seed_raises_during_capture(ups):
    from ups_b200 import _cabi as C
    from ups_b200.step import PartStep
    raw = _views(2, 32, 1)
    ups.make_tps(raw, CUB_TPS, seed=1)            # warm-up outside capture
    g = torch.cuda.CUDAGraph()
    with pytest.raises(C.UpsError, match="captured CUDA graph"):
        with torch.cuda.graph(g):
            ups.make_tps(raw, CUB_TPS, seed=1)
    d = cuda(make_inputs(2, 32, 16, 32, V=3, seed=1))
    st = PartStep(2, 32, 16, 32, n_views=3)
    st.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"], tps_seed=1)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(C.UpsError, match="captured CUDA graph"):
        with torch.cuda.graph(g):
            st.forward(d["views"], None, None, d["l0"], d["l1"], d["feat"], tps_seed=1)


# ---------------------------------------------------------------- g. opcheck, torch.compile
def test_opcheck(ups):
    from ups_b200 import ops
    s = ups.tps.draw_scalars(**CUB_TPS)
    dev = torch.device("cuda", torch.cuda.current_device())
    for args in ((ops.NOISE_INT, None, 77, 5, 6, 2, s, dev), (ops.NOISE_DEVICE, _seed_tensor(SEED), 0, 0, 7, 1, s, dev)):
        torch.library.opcheck(ops.tps_draw, args)


def test_torch_compile_fullgraph(ups):
    raw = _views(4, 64, 2)
    seed_t = _seed_tensor(SEED)

    def fn(v0, v1, v2, seed):
        return ups.make_tps([v0, v1, v2], CUB_TPS, seed=seed, sample_offset=8)

    torch._dynamo.reset()
    got = torch.compile(fn, fullgraph=True)(*raw, seed_t)
    want = fn(*raw, seed_t)
    for a, b in zip(got, want):
        assert_bitexact(a, b, "compiled make_tps")


# ---------------------------------------------------------------- h. errors
def test_errors(ups):
    from ups_b200 import _cabi as C
    raw = _views(2, 32, 3)
    with pytest.raises(ValueError, match="not both"):
        ups.tps.tps_parameters(4, seed=1, generator=torch.Generator(), **CUB_TPS)
    with pytest.raises(ValueError, match="not both"):
        ups.make_tps(raw, CUB_TPS, seed=1, generator=torch.Generator())
    with pytest.raises(ValueError, match="divisible"):
        ups.tps.tps_parameters(5, seed=1, views=2, **CUB_TPS)
    with pytest.raises(ValueError, match="rot_scal"):
        ups.make_tps(raw, dict(CUB_TPS, rot_scal=3.2), seed=1)
    with pytest.raises(C.UpsError, match="sample_offset"):
        ups.make_tps(raw, CUB_TPS, seed=1, sample_offset=-1)
    with pytest.raises(C.UpsError, match="sample_offset"):
        ups.tps.tps_parameters(4, seed=1, sample_offset=-2, **CUB_TPS)
