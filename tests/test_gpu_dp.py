"""-m gpu: the data-parallel wrapper (SURVEY.md 8e, App. D T4).

* the stand-in modules' kernels against their oracle (one GPU);
* DataParallelPartStep at world size 1 == PartStep, and its gradient buffer holds the stand-in gradients;
* T4 under NCCL with two ranks (skipped on a one-GPU box): the sharded step equals the single-GPU step on the
  concatenated batch bit for bit per sample, and the all-reduced buffer equals the mean of the per-rank buffers.
  The only analogue in the reference is the IMM baseline's host-side tower averaging
  (baselines/imm/imm/train/cnn_train_multi.py:75-118).
"""
import os
import socket

import pytest
import torch

from oracle import standin as OSI
from util import ATOL, RTOL, assert_close, cuda, make_inputs

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _own_error_atol(want32, want64):
    """north-star absolute tolerance + twice the fp32 oracle's own distance from the fp64 value of the same sum"""
    return ATOL + 2.0 * float((want32.double() - want64).abs().max())


@pytest.mark.parametrize("B,S,K,F", [(8, 128, 16, 64), (3, 96, 25, 64), (2, 64, 8, 16)])
def test_standin_modules_vs_oracle(B, S, K, F):
    from ups_b200 import _cabi as C
    g = torch.Generator().manual_seed(5)
    P = S * S
    pooled = torch.randn(B, K, 3, generator=g)
    dfeat = torch.randn(B, K, F, generator=g)
    feat = torch.randn(B, K, F, generator=g)
    labels = torch.randint(0, K, (B, S, S), generator=g, dtype=torch.int64)
    g_recon = torch.randn(B, S, S, 3, generator=g)
    Wlin, blin = torch.randn(3, F, generator=g), torch.randn(F, generator=g)
    Whead, bhead = torch.randn(F + K, 3, generator=g), torch.randn(3, generator=g)
    d = cuda(dict(pooled=pooled, dfeat=dfeat, feat=feat, labels=labels, g_recon=g_recon, Wlin=Wlin, blin=blin,
                  Whead=Whead, bhead=bhead))
    st = torch.cuda.current_stream().cuda_stream
    ws = torch.empty(C.lib.ups_standin_workspace_bytes(B, P, K, F), dtype=torch.uint8, device="cuda")
    # forward
    f = torch.empty(B, K, F, device="cuda")
    C.call("ups_standin_tail_fwd", d["pooled"].data_ptr(), d["Wlin"].data_ptr(), d["blin"].data_ptr(), f.data_ptr(), B, K, 3, F, st)
    assert_close(f, OSI.tail_fwd(pooled, Wlin, blin), "tail fwd")
    r = torch.empty(B, P, 3, device="cuda")
    C.call("ups_standin_head_fwd", d["labels"].data_ptr(), d["feat"].data_ptr(), d["Whead"].data_ptr(), d["bhead"].data_ptr(),
           r.data_ptr(), B, P, K, F, st)
    assert_close(r, OSI.head_fwd(labels, feat, Whead, bhead), "head fwd")
    # backward (weight gradients)
    gt = torch.empty(4 * F, device="cuda")
    C.call("ups_standin_tail_bwd", d["pooled"].data_ptr(), d["dfeat"].data_ptr(), gt.data_ptr(), B, K, 3, F, ws.data_ptr(),
           ws.numel(), st)
    w64 = OSI.tail_grads(pooled, dfeat, Wlin, blin)
    w32 = torch.cat([(pooled.reshape(-1, 3).t() @ dfeat.reshape(-1, F)).reshape(-1), dfeat.sum((0, 1))])
    assert_close(gt, w64, "tail grads", rtol=RTOL, atol=_own_error_atol(w32, w64))
    gh = torch.empty((F + K) * 3 + 3, device="cuda")
    C.call("ups_standin_head_bwd", d["g_recon"].data_ptr(), d["labels"].data_ptr(), d["feat"].data_ptr(), gh.data_ptr(), B, P, K, F,
           ws.data_ptr(), ws.numel(), st)
    torch.cuda.synchronize()
    h64 = OSI.head_grads(g_recon, labels, feat, Whead, bhead)
    h32 = _head_grads_fp32(g_recon, labels, feat, K)
    assert_close(gh, h64, "head grads", rtol=RTOL, atol=_own_error_atol(h32, h64))
    # deterministic: same bits on a second run
    gh2 = torch.empty_like(gh)
    C.call("ups_standin_head_bwd", d["g_recon"].data_ptr(), d["labels"].data_ptr(), d["feat"].data_ptr(), gh2.data_ptr(), B, P, K, F,
           ws.data_ptr(), ws.numel(), st)
    assert torch.equal(gh, gh2)


def _head_grads_fp32(g_recon, labels, feat, K):
    """the same gradient evaluated in fp32 in the oracle's own order (one_hot^T @ g, then feat^T @ R)"""
    B, _, F = feat.shape
    oh = torch.nn.functional.one_hot(labels.reshape(B, -1), K).float()
    R = oh.transpose(1, 2) @ g_recon.reshape(B, -1, 3)                 # [B,K,3]
    dW = torch.cat([(feat.transpose(1, 2) @ R).sum(0), R.sum(0)], 0)   # [(F+K),3]
    return torch.cat([dW.reshape(-1), R.sum((0, 1))])


def test_dp_world1_equals_partstep_and_holds_standin_grads():
    from ups_b200.dp import DataParallelPartStep
    from ups_b200.step import PartStep
    B, S, K, F, V = 4, 64, 16, 64, 3
    inp = make_inputs(B, S, K, F, V, seed=3)
    d = cuda(inp)
    c = d["cot"]
    ref = PartStep(B, S, K, F, n_views=V)
    o_ref = ref.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
    g_ref = ref.backward(c["g_inj"], c["g_parts"], c["g_pooled"], c["g_m0"], c["g_m1"])
    dp = DataParallelPartStep(B, S, K, F, n_views=V, n_grad_params=100_000, standin=True)
    assert dp.step.fuse_fwd
    assert dp.world == 1 and dp.reducer.transport == "none"
    g_recon = torch.randn(B, S, S, 3, generator=torch.Generator().manual_seed(1)).cuda()
    for _ in range(2):   # twice: the second forward waits on the first step's (empty) reduction
        o = dp.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
        g = dp.backward(c["g_inj"], c["g_parts"], c["g_pooled"], c["g_m0"], c["g_m1"], g_recon=g_recon)
    dp.wait_grads()
    torch.cuda.synchronize()
    for k in ("m0", "m1", "labels0", "parts", "pooled", "inj"):
        assert torch.equal(o[k], o_ref[k]), k
    for k in ("dl0", "dl1", "dfeat"):
        assert torch.equal(g[k], g_ref[k]), k
    h64 = OSI.head_grads(g_recon.cpu(), o_ref["labels0"].cpu(), inp["feat"], dp.mod.Whead.cpu(), dp.mod.bhead.cpu())
    assert_close(dp.grads_head, h64, "grads_head", atol=1e-4)
    t64 = OSI.tail_grads(o_ref["pooled"].cpu(), g_ref["dfeat"].cpu(), dp.mod.Wlin.cpu(), dp.mod.blin.cpu())
    assert_close(dp.grads_tail, t64, "grads_tail", atol=1e-4)
    used = dp.grads.clone()
    used[dp.head_off:dp.head_off + dp.mod.n_head] = 0
    used[dp.tail_off:dp.tail_off + dp.mod.n_tail] = 0
    assert float(used.abs().max()) == 0.0, "the padding of the gradient buffer stays zero"


def test_ops_run_on_a_non_current_device():
    """ADVICE r1: tensors on cuda:1 while cuda:0 is current must launch on cuda:1 (needs two GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import ups_b200
    from oracle import parts as OP
    from ups_b200.step import PartStep
    torch.cuda.set_device(0)
    x = torch.randn(2, 32, 32, 16, generator=torch.Generator().manual_seed(0))
    p = ups_b200.nn.softmax(x.to("cuda:1"))
    assert p.device.index == 1 and torch.equal(p.cpu().view(torch.int32), OP.softmax(x).view(torch.int32))
    B, S, K, F, V = 2, 64, 16, 64, 3
    inp = make_inputs(B, S, K, F, V, seed=0)
    d = {k: (v.to("cuda:1") if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    step = PartStep(B, S, K, F, n_views=V, device="cuda:1")
    out = step.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
    torch.cuda.synchronize(1)
    ref = PartStep(B, S, K, F, n_views=V, device="cuda:0")
    d0 = cuda(inp)
    out0 = ref.forward(d0["views"], d0["coord"], d0["t_vector"], d0["l0"], d0["l1"], d0["feat"])
    torch.cuda.synchronize(0)
    assert torch.cuda.current_device() == 0
    for k in ("m0", "labels0", "parts", "inj"):
        assert torch.equal(out[k].cpu(), out0[k].cpu()), k


# ------------------------------------------------------------------------------------------ T4 (two ranks, NCCL)
def _t4_worker(rank, world, port, q, allreduce):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                          LOCAL_RANK=str(rank))
        import sys
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        sys.path[:0] = [root, os.path.join(root, "tests")]
        import torch.distributed as dist
        from ups_b200.dp import DataParallelPartStep, init_from_env, shard_bounds
        from ups_b200.step import PartStep
        from util import cuda as to_cuda, make_inputs as mk
        r, local, w = init_from_env("nccl")
        dev = torch.device("cuda", local)
        GB, S, K, F, V = 6, 64, 16, 64, 3
        inp = mk(GB, S, K, F, V, seed=11)           # the same global batch on every rank
        lo, hi = shard_bounds(GB, r, w)
        Bl = hi - lo
        c = inp["cot"]
        g_recon = torch.randn(GB, S, S, 3, generator=torch.Generator().manual_seed(2))
        # TPS parameters are [2*GB,8,2] = (view 0 of every sample, then view 1): take the shard's rows of both halves
        def tps_rows(t):
            return torch.cat([t[lo:hi], t[GB + lo:GB + hi]]).contiguous()

        def shard_pm(t):   # part-major [K*GB,...] -> [K*Bl,...]
            return t.reshape(K, GB, *t.shape[1:])[:, lo:hi].reshape(K * Bl, *t.shape[1:]).contiguous()
        loc = dict(views=inp["views"][:, lo:hi].contiguous(), coord=tps_rows(inp["coord"]), t_vector=tps_rows(inp["t_vector"]),
                   l0=inp["l0"][lo:hi], l1=inp["l1"][lo:hi], feat=inp["feat"][lo:hi], g_inj=c["g_inj"][lo:hi],
                   g_parts=shard_pm(c["g_parts"]), g_pooled=c["g_pooled"][lo:hi], g_m0=c["g_m0"][lo:hi], g_m1=c["g_m1"][lo:hi],
                   g_recon=g_recon[lo:hi])
        loc = {k: v.to(dev).contiguous() for k, v in loc.items()}
        n_params = 1_000_000
        dp = DataParallelPartStep(Bl, S, K, F, n_views=V, n_grad_params=n_params, device=dev, allreduce=allreduce)
        # a rank-dependent pattern in the padding, so that the whole buffer (not only the stand-in heads) is checked
        pad = torch.arange(dp.grads.numel(), device=dev, dtype=torch.float32).mul_(1e-3).add_(float(r + 1))
        res = {}
        for it in range(3):
            dp.grads.copy_(pad)
            torch.cuda.synchronize(dev)
            dist.barrier()
            out = dp.forward(loc["views"], loc["coord"], loc["t_vector"], loc["l0"], loc["l1"], loc["feat"])
            grad = dp.backward(loc["g_inj"], loc["g_parts"], loc["g_pooled"], loc["g_m0"], loc["g_m1"], g_recon=loc["g_recon"])
            dp.wait_grads()
            torch.cuda.synchronize(dev)
        reduced = dp.grads.clone()
        # expected: the mean over ranks of (padding pattern with the rank's own stand-in gradients written at the bucket heads)
        # (this rank's own stand-in gradients recomputed with the same kernels, outside the wrapper)
        from ups_b200 import _cabi as C
        mine = pad.clone()
        st = torch.cuda.current_stream(dev).cuda_stream
        ws = torch.empty(C.lib.ups_standin_workspace_bytes(Bl, S * S, K, F), dtype=torch.uint8, device=dev)
        C.call("ups_standin_head_bwd", loc["g_recon"].data_ptr(), out["labels0"].data_ptr(), loc["feat"].data_ptr(),
               mine[dp.head_off:dp.head_off + dp.mod.n_head].data_ptr(), Bl, S * S, K, F, ws.data_ptr(), ws.numel(), st)
        C.call("ups_standin_tail_bwd", out["pooled"].data_ptr(), grad["dfeat"].data_ptr(),
               mine[dp.tail_off:dp.tail_off + dp.mod.n_tail].data_ptr(), Bl, K, 3, F, ws.data_ptr(), ws.numel(), st)
        gathered = [torch.empty_like(mine) for _ in range(w)]
        dist.all_gather(gathered, mine)
        want = torch.stack(gathered).double().mean(0)
        got = reduced.double() * dp.reducer.grad_scale
        rel = float(((got - want).abs() / want.abs().clamp(min=1e-3)).max())
        res["allreduce_rel_err"] = rel
        res["transport"] = dp.reducer.transport
        res["fallback_reason"] = dp.reducer.fallback_reason
        # path outputs of the shard == the single-GPU step on the whole batch, bit for bit per sample
        full = PartStep(GB, S, K, F, n_views=V, device=dev)
        dfull = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
        cf = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in c.items()}
        of = full.forward(dfull["views"], dfull["coord"], dfull["t_vector"], dfull["l0"], dfull["l1"], dfull["feat"])
        gf = full.backward(cf["g_inj"], cf["g_parts"], cf["g_pooled"], cf["g_m0"], cf["g_m1"])
        torch.cuda.synchronize(dev)
        same = {}
        for k in ("m0", "m1", "labels0", "pooled", "inj"):
            same[k] = bool(torch.equal(out[k], of[k][lo:hi]))
        same["warped"] = bool(torch.equal(out["warped"], of["warped"][:, lo:hi]))
        same["parts"] = bool(torch.equal(out["parts"], shard_pm(of["parts"])))
        for k in ("dl0", "dl1", "dfeat"):
            same[k] = bool(torch.equal(grad[k], gf[k][lo:hi]))
        res["same"] = same
        q.put((rank, res))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, {"error": repr(e), "trace": traceback.format_exc()}))


@pytest.mark.parametrize("allreduce", ["auto", "nccl"])
def test_t4_two_ranks_sharded_step_and_allreduce(allreduce):
    if torch.cuda.device_count() < 2:
        pytest.skip("T4 needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_t4_worker, args=(r, 2, port, q, allreduce)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
    for r in range(2):
        assert "error" not in res[r], res[r].get("trace")
        assert all(res[r]["same"].values()), (r, res[r]["same"])
        assert res[r]["allreduce_rel_err"] <= 1e-6, (r, res[r])
        if allreduce == "nccl":
            assert res[r]["transport"] == "nccl"
    print("T4 transports:", {r: (res[r]["transport"], res[r]["fallback_reason"]) for r in range(2)})


def test_dp_world1_padded_part_count():
    """The data-parallel wrapper with the reference's shipped n_parts = 25 (padded to 32 inside PartStep): same outputs as
    the plain step, stand-in gradients against the oracle."""
    from ups_b200.dp import DataParallelPartStep
    from ups_b200.step import PartStep
    B, S, K, F, V = 3, 64, 25, 64, 3
    inp = make_inputs(B, S, K, F, V, seed=4)
    d = cuda(inp)
    c = d["cot"]
    ref = PartStep(B, S, K, F, n_views=V)
    assert ref.Kp == 32
    o_ref = ref.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
    g_ref = ref.backward(c["g_inj"], c["g_parts"], c["g_pooled"], c["g_m0"], c["g_m1"])
    dp = DataParallelPartStep(B, S, K, F, n_views=V, n_grad_params=100_000, standin=True)
    g_recon = torch.randn(B, S, S, 3, generator=torch.Generator().manual_seed(1)).cuda()
    for _ in range(2):
        o = dp.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
        g = dp.backward(c["g_inj"], c["g_parts"], c["g_pooled"], c["g_m0"], c["g_m1"], g_recon=g_recon)
    dp.wait_grads()
    torch.cuda.synchronize()
    for k in ("m0", "m1", "labels0", "parts", "pooled", "inj"):
        assert torch.equal(o[k], o_ref[k]), k
    for k in ("dl0", "dl1", "dfeat"):
        assert torch.equal(g[k], g_ref[k]), k
    h64 = OSI.head_grads(g_recon.cpu(), o_ref["labels0"].cpu(), inp["feat"], dp.mod.Whead.cpu(), dp.mod.bhead.cpu())
    assert_close(dp.grads_head, h64, "grads_head", atol=1e-4)
    t64 = OSI.tail_grads(o_ref["pooled"].cpu(), g_ref["dfeat"].cpu(), dp.mod.Wlin.cpu(), dp.mod.blin.cpu())
    assert_close(dp.grads_tail, t64, "grads_tail", atol=1e-4)


def test_path_config_presets_make_steps():
    """configs.PathConfig: the reference's config keys (train_cub_subset_tps.yaml:19-20,132,139,187-194) -> a PartStep."""
    from ups_b200.configs import CUB_SHIPPED, PathConfig
    cfg = PathConfig.from_dict(dict(CUB_SHIPPED.to_dict(), batch_size=2, spatial_size=64, unknown_key=1))
    step = cfg.make_step()
    assert (step.B, step.S, step.K, step.F, step.V) == (2, 64, 25, 64, 3) and step.Kp == 32
    d = cuda(make_inputs(2, 64, 25, 64, 3, seed=1))
    out = step.forward(d["views"], d["coord"], d["t_vector"], d["l0"], d["l1"], d["feat"])
    assert out["m0"].shape == (2, 64, 64, 25) and out["labels0"].max().item() < 25
