"""The training step's sampled logits (MeanFieldDistribution.sample, cub/code/nn.py:1421-1427): three arms in one process,
alternated round by round on the same PartStep buffers.

  (a) plain   : today's step on given logits l0, l1
  (b) eps     : 2 x torch.randn + 2 x ups_mean_field_sample_fwd (l = mean + noise_level * eps), then the step on l
  (c) seed    : the step on the means with noise_seed: the draw is made in registers inside the fused kernels

Per arm: ms/step (median over rounds of CUDA-event timed windows), images/s and the algorithmic bytes of one step
computed from the shapes (arm b adds, per side, eps written by randn, mean + eps read and l written: 16 bytes per logit).
Also ups_normal_philox_fwd against torch.randn at the size of one side's logits.  Prints one JSON document (and writes it
to --out).  Usage: python scripts/bench_sampled_step.py [--rounds 7] [--steps 20] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)

CASES = [  # name, S, K, F, V, B, TPS ranges
    ("cub_b256_k16", 128, 16, 64, 3, 256, "cub"),
    ("cub_b256_k25", 128, 25, 64, 3, 256, "cub"),
    ("pennaction_b512_k16", 128, 16, 64, 2, 512, "penn"),
]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 - recorded, not fatal
        q = f"nvidia-smi unavailable: {e!r}"
    return q


def timed(torch, fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def median(v):
    s = sorted(v)
    return s[len(s) // 2]


def run_case(torch, ups, C, name, S, K, F, V, B, tps, rounds, steps, warmup, level=1.0, seed=20261020):
    from ups_b200.configs import CUB_TPS, PENN_TPS
    from ups_b200.step import PartStep
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    P = S * S
    views = torch.rand(V, B, S, S, 3, device=dev, generator=g) * 2 - 1
    l0, l1 = torch.randn(B, S, S, K, device=dev, generator=g), torch.randn(B, S, S, K, device=dev, generator=g)
    feat = torch.randn(B, K, F, device=dev, generator=g)
    cot = dict(g_inj=torch.randn(B, S, S, F + K, device=dev, generator=g), g_parts=torch.randn(K * B, S, S, 3, device=dev, generator=g),
               g_pooled=torch.randn(B, K, 3, device=dev, generator=g), g_m0=torch.randn(B, S, S, K, device=dev, generator=g),
               g_m1=torch.randn(B, S, S, K, device=dev, generator=g))
    prm = ups.tps_parameters(2 * B, generator=torch.Generator().manual_seed(1234), device=dev,
                             **(CUB_TPS if tps == "cub" else PENN_TPS))
    coord, tv = ups.make_input_tps_param(prm)
    step = PartStep(B, S, K, F, n_views=V)
    eps0, eps1 = torch.empty_like(l0), torch.empty_like(l1)
    s0, s1 = torch.empty_like(l0), torch.empty_like(l1)
    n = l0.numel()
    gen = torch.Generator(device=dev).manual_seed(seed)

    def bwd():
        step.backward(cot["g_inj"], cot["g_parts"], cot["g_pooled"], cot["g_m0"], cot["g_m1"])

    def plain():
        step.forward(views, coord, tv, l0, l1, feat)
        bwd()

    def eps_arm():
        st = torch.cuda.current_stream().cuda_stream
        torch.randn(l0.shape, generator=gen, device=dev, out=eps0)
        torch.randn(l1.shape, generator=gen, device=dev, out=eps1)
        C.call("ups_mean_field_sample_fwd", l0.data_ptr(), eps0.data_ptr(), level, s0.data_ptr(), n, st)
        C.call("ups_mean_field_sample_fwd", l1.data_ptr(), eps1.data_ptr(), level, s1.data_ptr(), n, st)
        step.forward(views, coord, tv, s0, s1, feat)
        bwd()

    def seed_arm():
        step.forward(views, coord, tv, l0, l1, feat, noise_seed=seed, noise_level=level)
        bwd()

    arms = dict(plain=plain, eps=eps_arm, seed=seed_arm)
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(timed(torch, fn, steps))
    step_bytes = step.algorithmic_bytes_per_image() * B
    extra = 2 * 16 * n                 # per side: randn writes eps, the sample reads mean + eps and writes l
    res = {}
    for k in arms:
        m = median(ms[k])
        b = step_bytes + (extra if k == "eps" else 0)
        res[k] = dict(ms_per_step=round(m, 4), img_per_s=round(B / m * 1e3, 1), bytes_per_step=b,
                      gb_per_s=round(b / m / 1e6, 1), ms_rounds=[round(x, 4) for x in ms[k]])
    # the draw alone, one side's logits: ups_normal_philox_fwd vs torch.randn (write-only, 4 bytes per value)
    out = torch.empty(B * P, K, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    draw = lambda: C.call("ups_normal_philox_fwd", seed, 0, 0, B * P, K, out.data_ptr(), st)  # noqa: E731
    rnd = lambda: torch.randn(out.shape, generator=gen, device=dev, out=out)  # noqa: E731
    for _ in range(warmup):
        draw()
        rnd()
    dr, rn = [], []
    for _ in range(rounds):
        dr.append(timed(torch, draw, steps))
        rn.append(timed(torch, rnd, steps))
    standalone = dict(n_values=B * P * K, bytes=4 * B * P * K,
                      ups_normal_philox_fwd_ms=round(median(dr), 4), torch_randn_ms=round(median(rn), 4),
                      ups_normal_philox_fwd_gb_per_s=round(4 * B * P * K / median(dr) / 1e6, 1),
                      torch_randn_gb_per_s=round(4 * B * P * K / median(rn) / 1e6, 1))
    del step
    torch.cuda.empty_cache()
    return dict(case=name, S=S, K=K, F=F, V=V, B=B, noise_level=level, arms=res, standalone_draw=standalone,
                seed_vs_eps_speedup=round(res["eps"]["ms_per_step"] / res["seed"]["ms_per_step"], 3),
                seed_vs_plain_ratio=round(res["seed"]["ms_per_step"] / res["plain"]["ms_per_step"], 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_sampled_step.py measures on the GPU; there is no CPU path"
    import ups_b200 as ups
    from ups_b200 import _cabi as C
    want = set(args.cases.split(","))
    doc = dict(card=card(), device=torch.cuda.get_device_name(0), library=C.version(), rounds=args.rounds, steps=args.steps,
               cases=[])
    for c in CASES:
        if c[0] in want:
            doc["cases"].append(run_case(torch, ups, C, *c, rounds=args.rounds, steps=args.steps, warmup=args.warmup))
            print(json.dumps(doc["cases"][-1]), flush=True)
    doc["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(dict(card=doc["card"], device=doc["device"])))


if __name__ == "__main__":
    main()
