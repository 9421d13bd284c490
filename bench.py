#!/usr/bin/env python
"""Benchmark of the per-step part-disentanglement path (BASELINE.json metric:
part-step images/sec, forward + backward, and fraction of the HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cub|deepfashion|pennaction]
    python bench.py --impl reference ...      # the CPU restatement of the reference path, host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs to DIR/<name>.npy

One "step" = forward + backward of the path (TPS warp of the views, part softmax, masks and
labels, mask_parts + pooling, unpool + inject, and the backward of all of it) on one batch of
synthetic inputs.  Prints ONE JSON line on rank 0.  Writes nothing into the source tree (the
tree may be read-only): no bytecode caches either.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (spatial, K, F, views, per-GPU batch, tps ranges)  — BASELINE.json configs[1..3]
    "cub": dict(S=128, K=16, F=64, V=3, B=256, use_tps=True,
                desc="CUB 128x128, K=16, F=64, 3 warped views, batch 256 per GPU (BASELINE.json configs[1])"),
    "deepfashion": dict(S=256, K=16, F=64, V=2, B=128, use_tps=True,
                        desc="DeepFashion 256x256, K=16, F=64, 2 warped views, batch 128 per GPU (configs[2])"),
    "pennaction": dict(S=128, K=16, F=64, V=2, B=512, use_tps=True,
                       desc="PennAction 128x128, K=16, F=64, 2 per-sample warps, batch 512 per GPU (configs[3])"),
}
CPU_SAMPLE_B = 8   # BASELINE.json configs[0]: batch 8 on the host CPU


_JSON_OUT = None


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_port_rate(wl, steps, warmup, threads=None):
    """fwd+bwd of the oracle (CPU restatement of the reference path) on a bounded sample."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))      # the CPU arm is the one place bench.py uses the checker's helpers
    from oracle import step as OS
    from util import make_inputs
    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = CPU_SAMPLE_B
    inp = make_inputs(B, wl["S"], wl["K"], wl["F"], wl["V"], seed=0)
    cot = dict(inp["cot"], g_warped=None)
    views = [v for v in inp["views"]]

    def one():
        OS.step_forward_backward(views, inp["coord"], inp["t_vector"], inp["l0"], inp["l1"], inp["feat"], cot,
                                 use_tps=wl["use_tps"])
    for _ in range(warmup):
        one()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return B / med, med, cores, f"{steps} fwd+bwd steps of batch {B} at the workload's resolution (median), {cores} torch threads"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    # one step = one fwd+bwd of a bounded sample (batch 8, ~0.7 s on 16 cores)
    steps, warm = args.steps, args.warmup
    rate, med, cores, sample = cpu_port_rate(wl, steps, warm)
    line = {
        "impl": "reference", "metric": "part-step images/sec (fwd+bwd)", "value": rate, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": med * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "sample_batch": CPU_SAMPLE_B},
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU restatement (oracle/) of the reference's TF-1.14 op chain; TF itself is not installable here",
    }
    emit(line)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Polls NVML (SM clock, throttle reasons) every few ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.004)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------ GPU arm
def base_call(name):
    """The C-ABI call without the suffix of its argument form: `ups_step_decode_bwd_tc_rows` (row-length argument) and
    `ups_step_encode_fwd_planes` (part-plane count) launch the same kernels as the plain entry points."""
    for suffix in ("_rows", "_planes"):
        if name.endswith(suffix):
            return name[:-len(suffix)]
    return name


def call_bytes(name, K, F, V, B, P):
    """Algorithmic (compulsory) bytes of one C-ABI call of the step, fp32, K parts, F features, 3 channels; None if the
    call is not one of the path kernels.  Per decode/encode pixel there are B*P pixels, per warped pixel V*B*P."""
    name = base_call(name)
    warp_px, px = V * B * P, B * P
    per = {
        "ups_tps_warp_fwd": (4 * (3 + 3), warp_px), "ups_tps_warp_pair_fwd": (4 * (3 + 3), warp_px),
        "ups_tps_warp_bwd": (4 * (3 + 3), warp_px), "ups_tps_warp_pair_bwd": (4 * (3 + 3), warp_px),
        "ups_tps_warp_bwd_sum": (4 * (3 + 3) * V + 4 * 3, px),  # + the encode side's dimg1, added on the fly (view 1)
        "ups_step_encode_fwd": (4 * (K + 3 + K + 3 * K), px),
        "ups_step_decode_fwd": (4 * (K + K + 2 + F + K), px),
        "ups_step_decode_bwd": (4 * ((F + K) + K + K + K), px), "ups_step_decode_bwd_tc": (4 * ((F + K) + K + K + K), px),
        "ups_step_encode_bwd": (4 * (3 * K + 3 + K + K + K), px),
        # K1 + K3 in one launch: the decode side's bytes per pixel plus V warped pixels of 24 bytes
        "ups_step_warp_decode_fwd": (4 * (K + K + 2 + F + K) + V * 4 * (3 + 3), px),
    }
    if name not in per:
        return None
    b, n = per[name]
    return b * n


CALL_KERNEL = {  # C-ABI call -> the kernel that dominates it (profiles/ncu_traffic.json keys)
    "ups_tps_warp_fwd": "tps_warp_fwd_kernel", "ups_tps_warp_pair_fwd": "tps_warp_fwd_kernel",
    "ups_step_encode_fwd": "step_encode_fwd_kernel", "ups_step_decode_fwd": "step_decode_fwd_kernel",
    "ups_step_decode_bwd": "step_decode_bwd_kernel", "ups_step_decode_bwd_tc": "step_decode_bwd_tma_kernel",
    "ups_step_encode_bwd": "step_encode_bwd_kernel", "ups_step_warp_decode_fwd": "step_warp_decode_fwd_kernel",
    "ups_tps_warp_bwd": "tps_warp_bwd_kernel", "ups_tps_warp_bwd_sum": "tps_warp_bwd_kernel",
}


def ncu_traffic(call, workload, B):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    if d.get("workload") != workload or d.get("B") != B:
        return None, None
    return d["bytes_per_launch"].get(CALL_KERNEL.get(base_call(call), "")), d.get("source")


def set_rank_affinity(local, world_local):
    """Give every rank its own slice of the host cores BEFORE it allocates pinned memory (first touch) and starts its
    helper threads: eight ranks that all float over all cores (the box reports one NUMA node, CPU affinity 0-31 for
    every GPU) contend for the same cores with their launch, NCCL-proxy and clock-sampler threads.  Returns the cores."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if world_local <= 1 or len(cores) < 2 * world_local:
            return cores
        per = len(cores) // world_local
        mine = cores[local * per:(local + 1) * per]
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:  # noqa: BLE001 - affinity is an optimisation, never a requirement
        return None


def make_workload_tensors(torch, ups_b200, wl, name, B, dev, rank, seed, tps_bwd):
    from ups_b200.configs import CUB_TPS, PENN_TPS
    from ups_b200.dp import rank_seed
    S, K, F, V = wl["S"], wl["K"], wl["F"], wl["V"]
    g = torch.Generator(device=dev).manual_seed(rank_seed(seed, rank))
    t = dict(
        views=torch.rand(V, B, S, S, 3, device=dev, generator=g) * 2 - 1,
        l0=torch.randn(B, S, S, K, device=dev, generator=g), l1=torch.randn(B, S, S, K, device=dev, generator=g),
        feat=torch.randn(B, K, F, device=dev, generator=g), g_inj=torch.randn(B, S, S, F + K, device=dev, generator=g),
        g_parts=torch.randn(K * B, S, S, 3, device=dev, generator=g), g_pooled=torch.randn(B, K, 3, device=dev, generator=g),
        g_m0=torch.randn(B, S, S, K, device=dev, generator=g), g_m1=torch.randn(B, S, S, K, device=dev, generator=g),
        g_recon=torch.randn(B, S, S, 3, device=dev, generator=g),
        g_warped=torch.randn(V, B, S, S, 3, device=dev, generator=g) if tps_bwd else None)
    tps_kw = CUB_TPS if name == "cub" else PENN_TPS
    prm = ups_b200.tps_parameters(2 * B, generator=torch.Generator().manual_seed(1234 + rank), device=dev, **tps_kw)
    t["coord"], t["tv"] = ups_b200.make_input_tps_param(prm)
    return t


DUMP_BYTES = 60_000_000    # --dump-outputs: data budget of all arrays together, under 64 MB with the .npy headers


def dump_outputs(out_dir, outputs):
    """Write the arrays of `outputs` (name -> tensor) as out_dir/<name>.npy: float32, or float64 for integer arrays
    (the labels).  An array with more elements than its share of DUMP_BYTES is written as a 1-D sample of its flat
    entries, at positions drawn by a generator seeded with 0: they depend on the array's size only, so two runs or
    two builds sample the same entries."""
    import numpy as np
    import torch
    arrays = {k: v for k, v in outputs.items() if v is not None}
    cap = DUMP_BYTES // (8 * max(1, len(arrays)))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in sorted(arrays.items()):
        if t.numel() > cap:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), size=cap))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        a = a.astype(np.float64 if np.issubdtype(a.dtype, np.integer) else np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_workload(args, torch, dist, ups_b200, name, B, dev, rank, world, reducer, steps, warmup, detailed,
                     dump_dir=None):
    """K timed steps of the data-parallel part step on workload `name` with inputs resident in HBM.
    Returns (record, dp, tensors); `detailed` adds per-call CUDA events and the launch count.  `dump_dir`: rank 0
    writes what forward and backward returned in the last timed step there (dump_outputs)."""
    from ups_b200 import _cabi as C
    from ups_b200.dp import DataParallelPartStep
    wl = dict(WORKLOADS[name])
    if args.n_parts:
        wl["K"] = args.n_parts
        wl["desc"] = wl["desc"].replace("K=16", "K=%d" % args.n_parts)
    S, K, F, V = wl["S"], wl["K"], wl["F"], wl["V"]
    P = S * S
    dp = DataParallelPartStep(B, S, K, F, n_views=V, use_tps=wl["use_tps"], views_grad=args.tps_bwd, device=dev,
                              decode_bwd=args.decode_bwd, reducer=reducer)
    step = dp.step
    t = make_workload_tensors(torch, ups_b200, wl, name, B, dev, rank, args.seed, args.tps_bwd)
    last = {}    # what the last step's forward and backward returned (views of the step's output buffers)

    def one_step():
        last.update(dp.forward(t["views"], t["coord"], t["tv"], t["l0"], t["l1"], t["feat"]))
        last.update(dp.backward(t["g_inj"], t["g_parts"], t["g_pooled"], t["g_m0"], t["g_m1"], t["g_warped"],
                                g_recon=t["g_recon"]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        one_step()
    barrier()

    # ---- timed region: exactly `steps` steps, device time; per-call events on the launching stream
    marks = []
    raw_call = C.call

    def timed_call(cname, *a):
        if cname.startswith("ups_dp_"):     # enqueued on the reducer's side stream, not timed per call
            return raw_call(cname, *a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        raw_call(cname, *a)
        e1.record()
        marks.append((cname, e0, e1))

    sampler = ClockSampler(dev.index) if detailed else None
    if sampler:
        sampler.start()
    C.launch_count_reset()
    if detailed:
        C.call = timed_call
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for _ in range(steps):
        one_step()
    dp.wait_grads()            # the last step's gradient buckets are part of the last step
    t1.record()
    barrier()
    C.call = raw_call
    launches = C.launch_count()
    clocks = sampler.stop() if sampler else None
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, last)
    ms = t0.elapsed_time(t1)
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    ms_per_step = ms / steps
    peak, peak_src = load_peaks()
    step_bytes = step.algorithmic_bytes_per_image() * B
    step_gbs = step_bytes / (ms_per_step * 1e-3) / 1e9
    rec = {"value": world * B * steps / (ms * 1e-3), "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup,
           "per_gpu_batch": B, "workload": wl["desc"],
           "step_roofline": {"algorithmic_bytes_per_image": step.algorithmic_bytes_per_image(), "achieved": step_gbs,
                             "peak": peak, "unit": "GB/s", "frac": step_gbs / peak, "frac_of_nominal_8TBs": step_gbs / 8000.0},
           "gpu_launches": launches, "clocks": clocks}
    if detailed:
        per_call = {}
        for cname, e0, e1 in marks:
            per_call.setdefault(cname, []).append(e0.elapsed_time(e1))
        call_ms = {n: sum(v) / steps for n, v in per_call.items()}
        dom = max(call_ms, key=call_ms.get)
        dom_bytes = call_bytes(dom, K, F, V, B, P)
        n_dom = len(per_call[dom]) / steps
        dom_launch_ms = call_ms[dom] / n_dom
        achieved = (dom_bytes / n_dom) / (dom_launch_ms * 1e-3) / 1e9 if dom_bytes else None
        traffic, traffic_src = ncu_traffic(dom, name, B)
        rec["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                           "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                           "traffic_source": traffic_src, "peak_source": peak_src,
                           "algorithmic_bytes_per_launch": dom_bytes / n_dom if dom_bytes else None,
                           "launch_ms": dom_launch_ms}
        rec["per_call_ms"] = {k: round(v, 4) for k, v in sorted(call_ms.items())}
        rec["per_call_frac_of_hbm"] = {k: round(call_bytes(k, K, F, V, B, P) / (v * 1e-3) / 1e9 / peak, 4)
                                       for k, v in sorted(call_ms.items()) if call_bytes(k, K, F, V, B, P) and v > 0}
    return rec, dp, t


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import ups_b200
    from ups_b200.dp import GradAllReducer, init_from_env, two_buckets

    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
    cores = set_rank_affinity(int(os.environ.get("LOCAL_RANK", "0")), local_world) if not args.no_affinity else None
    rank, local, world = init_from_env()
    assert world == args.gpus or world == 1, (world, args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if cores:
        torch.set_num_threads(max(1, min(len(cores), 8)))
    wl = dict(WORKLOADS[args.workload])
    if args.n_parts:
        wl["K"] = args.n_parts
        wl["desc"] = wl["desc"].replace("K=16", "K=%d" % args.n_parts)
    S, K, F, V, B = wl["S"], wl["K"], wl["F"], wl["V"], args.batch or wl["B"]
    # one flat gradient buffer (symmetric memory when N>1) shared by every workload measured in this process
    n_grad = (int(args.grad_mb * 1e6 / 4) + 3) // 4 * 4
    from ups_b200.dp import default_allreduce_ctas
    reducer = GradAllReducer(n_grad, dev, buckets=two_buckets(n_grad), impl=args.allreduce,
                             n_ctas=args.allreduce_ctas or default_allreduce_ctas(world))
    warm = max(args.warmup, 3)
    rec, dp, t = measure_workload(args, torch, dist, ups_b200, args.workload, B, dev, rank, world, reducer, args.steps, warm,
                                  detailed=True, dump_dir=args.dump_outputs)
    step = dp.step
    line = {
        "metric": "part-step images/sec (fwd+bwd)", "value": rec["value"], "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "per_gpu_batch": B, "global_batch": B * world, "spatial": S, "n_parts": K,
                   "local_app_size": F, "views": V, "tps_backward": bool(args.tps_bwd), "decode_bwd": step.decode_bwd,
                   "parallelism": f"dp{world} (batch-sharded; no data-path collective; {reducer.flat.numel() * 4 / 1e6:.0f} MB fp32 "
                                  f"gradient mean per step in two buckets, fed by the stand-in gradient kernels, when N>1)",
                   "allreduce": {"transport": reducer.transport, "impl": reducer.impl, "ctas": reducer.n_ctas,
                                 "fallback_reason": reducer.fallback_reason,
                                 "buckets_mb": [round(n * 4 / 1e6, 1) for _, n in reducer.bounds]},
                   "host_cores_of_rank": (len(cores) if cores else None),
                   "l2": "inputs larger than L2: one step touches %.1f GB per GPU (L2 = 126 MB)"
                         % (step.algorithmic_bytes_per_image() * B / 1e9)},
        "clocks": rec["clocks"],
        "gpu_launches": rec["gpu_launches"],
        "roofline": rec["roofline"],
        "step_roofline": rec["step_roofline"],
        "per_call_ms": rec["per_call_ms"],
        "per_call_frac_of_hbm": rec["per_call_frac_of_hbm"],
    }

    # ---- e2e: same metric through the public API with HOST buffers (pinned), copies in the timed region
    if not args.no_e2e:
        targs = dict(views=t["views"], coord=t["coord"].cpu(), tv=t["tv"].cpu(), l0=t["l0"], l1=t["l1"], feat=t["feat"],
                     g_inj=t["g_inj"], g_parts=t["g_parts"], g_pooled=t["g_pooled"], g_m0=t["g_m0"], g_m1=t["g_m1"],
                     g_warped=t["g_warped"], g_recon=t["g_recon"])
        line["e2e"] = run_e2e(args, torch, dist, dp, dev, world, targs, B)
        # same step with the views crossing PCIe as the dataset's uint8 pixels (reported beside, not instead of, e2e)
        line["e2e_uint8_views"] = run_e2e(args, torch, dist, dp, dev, world, targs, B, u8=True)

    # ---- BASELINE.json configs[2], configs[3] at this N (the other workloads, device-resident, fewer steps)
    if not args.no_scale_workloads:
        del dp, t, step
        torch.cuda.empty_cache()
        line["scale_workloads"] = {}
        for other in sorted(WORKLOADS):
            if other == args.workload:
                continue
            try:
                r2, dp2, t2 = measure_workload(args, torch, dist, ups_b200, other, WORKLOADS[other]["B"], dev, rank, world,
                                               reducer, max(5, min(args.steps, 20)), 3, detailed=False)
                line["scale_workloads"][other] = {
                    "value": r2["value"], "unit": "images/s", "ms_per_step": r2["ms_per_step"], "steps": r2["steps"],
                    "per_gpu_batch": r2["per_gpu_batch"], "global_batch": r2["per_gpu_batch"] * world,
                    "workload": r2["workload"], "step_roofline_frac": r2["step_roofline"]["frac"],
                    "step_roofline_frac_of_nominal_8TBs": r2["step_roofline"]["frac_of_nominal_8TBs"]}
                del dp2, t2
            except Exception as e:  # noqa: BLE001 - a secondary workload must never cost the headline line
                line["scale_workloads"][other] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N=1 only): the oracle on the host cores, bounded sample
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, med, ncores, sample = cpu_port_rate(wl, steps=5, warmup=1)
        line["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": ncores, "kind": "port", "sample": sample}
    # ---- SURVEY.md 8f N4 (next row): the first decoder / encoder convolutions on the part assignment, per C-ABI
    # call with CUDA events, L2 flushed between calls; the library (cuDNN) legs on the materialised tensors beside them
    if rank == 0 and world == 1 and args.workload == "cub" and not args.no_n4:
        try:
            torch.cuda.empty_cache()
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import bench_inject_conv
            n4 = bench_inject_conv.measure(B, S, K, library=True, iters=5)
            line["n4_first_conv"] = {"shape": n4["shape"], "l2": n4["l2"],
                                     "calls": {k: ({"ms": round(v["ms"], 4), "frac_of_measured_hbm": round(v["frac_of_measured_hbm"], 4)}
                                                   if "ms" in v else v) for k, v in n4["calls"].items()}}
            del n4
            torch.cuda.empty_cache()
            fs = bench_inject_conv.measure_folded_step(B, S, K, iters=5)
            lib = {k: v["ms"] for k, v in line["n4_first_conv"]["calls"].items() if k.startswith("library")}
            line["n4_first_conv"]["folded_step"] = dict(
                fs, library_path_ms_per_step=(rec["ms_per_step"] + sum(lib.values())) if lib else None,
                library_path="the path step above (inj and parts materialised) + the four cuDNN legs (conv fwd / bwd on "
                             "injected and on the part images)")
        except Exception as e:  # the N4 leg must never cost the headline line
            line["n4_first_conv"] = {"error": repr(e)[:300]}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, torch, dist, dp, dev, world, t, B, u8=False):
    """Host-resident per-step inputs (what the reference feeds through feed_dict each step: the
    image views, cub/code/SB_model48i/model.py:316-327, plus the TPS parameters drawn on the host)
    are copied host->device every step from pinned memory; the step's host-visible results (the
    int64 part labels that evaluation consumes, the pooled part appearances and dfeat) are read
    back every step.  Logits, part features and cotangents are produced ON the device by the
    CNNs that surround the path in the real model, so they stay device-resident here too.
    Copies run on a side stream, double-buffered, so that they overlap the previous step.

    u8=True: the views cross PCIe as the dataset's uint8 pixels and the data pipeline's
    `astype(float32) * 2 / 255 - 1` (cub/code/data/data.py:134) runs on the device inside
    PartStep.forward (ups_views_u8_to_f32) -- same step, a quarter of the H2D bytes."""
    if u8:
        g = torch.Generator().manual_seed(args.seed)
        views_h = torch.randint(0, 256, tuple(t["views"].shape), dtype=torch.uint8, generator=g).pin_memory()
    else:
        views_h = t["views"].cpu().pin_memory()
    coord_h, tv_h = t["coord"].pin_memory(), t["tv"].pin_memory()
    step = dp.step
    # u8 leg: the label map is read back at one byte per pixel too (ups_labels_i64_to_u8; n_parts <= 255)
    lab_dtype = torch.uint8 if u8 else torch.int64
    lab_h = torch.empty(step.labels0.shape, dtype=lab_dtype).pin_memory()
    pooled_h = torch.empty(step.pooled.shape).pin_memory()
    dfeat_h = torch.empty(step.dfeat.shape).pin_memory()
    lab_d = torch.empty(step.labels0.shape, dtype=lab_dtype, device=dev)
    pooled_d, dfeat_d = (torch.empty_like(x) for x in (step.pooled, step.dfeat))
    bufs = [dict(views=torch.empty(views_h.shape, dtype=views_h.dtype, device=dev),
                 coord=torch.empty(coord_h.shape, device=dev),
                 tv=torch.empty(tv_h.shape, device=dev)) for _ in range(2)]
    copy_s = torch.cuda.Stream(device=dev)
    out_s = torch.cuda.Stream(device=dev)
    main_s = torch.cuda.current_stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    done = torch.cuda.Event()
    drained = torch.cuda.Event()
    h2d = views_h.numel() * views_h.element_size() + coord_h.numel() * 4 + tv_h.numel() * 4
    d2h = lab_h.numel() * lab_h.element_size() + pooled_h.numel() * 4 + dfeat_h.numel() * 4

    def stage(i):
        b = bufs[i % 2]
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(freed[i % 2])
            b["views"].copy_(views_h, non_blocking=True)
            b["coord"].copy_(coord_h, non_blocking=True)
            b["tv"].copy_(tv_h, non_blocking=True)
            ready[i % 2].record(copy_s)

    def run(n):
        for ev in freed:
            ev.record(main_s)
        drained.record(main_s)
        stage(0)
        for i in range(n):
            if i + 1 < n:
                stage(i + 1)
            b = bufs[i % 2]
            main_s.wait_event(ready[i % 2])
            dp.forward(b["views"], b["coord"], b["tv"], t["l0"], t["l1"], t["feat"])
            dp.backward(t["g_inj"], t["g_parts"], t["g_pooled"], t["g_m0"], t["g_m1"], t["g_warped"], g_recon=t["g_recon"])
            freed[i % 2].record(main_s)
            # results -> a device staging copy (35 MB device-to-device, ~12 us), read back from there on
            # its own stream: the D2H of step i overlaps the kernels of step i+1
            main_s.wait_event(drained)          # the previous read-back has left the staging buffers
            lab_d.copy_(step.labels_u8() if u8 else step.labels0, non_blocking=True)
            pooled_d.copy_(step.pooled, non_blocking=True)
            dfeat_d.copy_(step.dfeat, non_blocking=True)
            done.record(main_s)
            with torch.cuda.stream(out_s):
                out_s.wait_event(done)
                lab_h.copy_(lab_d, non_blocking=True)
                pooled_h.copy_(pooled_d, non_blocking=True)
                dfeat_h.copy_(dfeat_d, non_blocking=True)
                drained.record(out_s)
        dp.wait_grads()
        main_s.wait_event(drained)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run(3)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = max(5, min(args.steps, 50))
    t0.record()
    run(n)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    assert int(lab_h.max()) < dp.step.K
    return {"value": world * B * n / (ms * 1e-3), "unit": "images/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "steps": n, "ms_per_step": ms / n,
            "h2d_GBs_per_rank": h2d / (ms / n * 1e-3) / 1e9, "d2h_GBs_per_rank": d2h / (ms / n * 1e-3) / 1e9,
            "boundary": ("host: %s views + TPS params in, %s labels + pooled + dfeat out; "
                         "logits/features/cotangents device-resident (CNN outputs in the real model)")
                        % (("uint8 (normalised on the device as cub/code/data/data.py:134 does on the host)", "uint8") if u8
                           else ("fp32", "int64"))}


def main():
    # stdout carries exactly one JSON line: everything else that writes to file descriptor 1 (NCCL prints its
    # version banner there when the box sets NCCL_DEBUG) is sent to stderr; the line goes out through the saved descriptor
    global _JSON_OUT
    sys.dont_write_bytecode = True      # the modules imported from here on leave no __pycache__ in the tree
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cub", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override")
    ap.add_argument("--n-parts", type=int, default=0, help="part count override (e.g. 25, the reference's shipped n_parts)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--tps-bwd", action="store_true", help="also back-propagate into the input views (K6)")
    ap.add_argument("--decode-bwd", default="auto", choices=["auto", "tc", "simt"],
                    help="K4 variant: tcgen05 tensor-core kernel or CUDA-core kernel")
    ap.add_argument("--grad-mb", type=float, default=133.2,
                    help="size of the stand-in encoder/decoder gradient buffer all-reduced per step when N>1 "
                         "(33.3 M fp32 parameters of the reference's CNNs, SURVEY.md section 2)")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "peer", "nccl"],
                    help="gradient mean when N>1: ups_dp_allreduce over symmetric memory (multicast / peer) or ncclAllReduce")
    ap.add_argument("--allreduce-ctas", type=int, default=0, help="CTAs of the all-reduce kernel (0: by world size)")
    ap.add_argument("--no-scale-workloads", action="store_true", help="skip the DeepFashion / PennAction legs")
    ap.add_argument("--no-affinity", action="store_true", help="do not give each rank its own slice of the host cores")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-n4", action="store_true", help="skip the N4 first-convolution microbenchmark leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what forward and backward returned in the last one as DIR/<name>.npy "
                         "(float32; integer outputs as float64; arrays too large for 64 MB in all as a fixed seeded "
                         "sample of their entries; rank 0's shard when N>1)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
