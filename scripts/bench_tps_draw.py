"""The TPS warp parameters drawn on the host (tps_parameters from a torch.Generator, then six host-to-device copies) and
on the device from a seed (ups::tps_draw: the draw, make_input_tps_param and the solve in one launch).

  (1) model.make_tps at CUB B=256 S=128, three views: generator, int seed, one-element int64 CUDA seed.  CUDA-event time
      and wall-clock time (a host clock around the same window, ending in a synchronize): the host draw and its copies
      show up in wall-clock time only.
  (2) one training step of a tiny model in the reference's order (make_tps -> e_pi -> part_encode -> e_alpha ->
      part_decode -> dd, reconstruction + categorical KL loss, backward) at CUB_SHIPPED (B=8 S=128 K=25 F=64), with a
      device seed for the warp and the logit noise: eager against one captured CUDA graph of the whole step.  Only the
      device seed makes the graph possible: a host draw would be frozen into it.
  (3) PartStep forward + backward at CUB B=256 S=128 K=16 F=64, three views: given coord / t_vector against tps_seed.

Arms alternate within each round; times are medians over rounds, with the range over rounds.  Prints one JSON document
with the card's name and power limit (and writes it to --out).
Usage: python scripts/bench_tps_draw.py [--rounds 7] [--steps 20] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 - recorded, not fatal
        q = f"nvidia-smi unavailable: {e!r}"
    return q


def timed(torch, fn, steps):
    """(CUDA-event ms, wall-clock ms) per step over one window that ends in a synchronize."""
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps, (time.perf_counter() - t0) * 1e3 / steps


def summary(v):
    s = sorted(v)
    return dict(median=s[len(s) // 2], min=s[0], max=s[-1])


def run_arms(torch, arms, rounds, steps, warmup):
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    res = {k: ([], []) for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ev, wall = timed(torch, fn, steps)
            res[k][0].append(ev)
            res[k][1].append(wall)
    return {k: dict(event_ms=summary(e), wall_ms=summary(w)) for k, (e, w) in res.items()}


def make_tps_arms(torch, M, configs):
    B, S = 256, 128
    g = torch.Generator(device="cuda").manual_seed(0)
    views = [torch.rand(B, S, S, 3, device="cuda", generator=g) * 2 - 1 for _ in range(3)]
    kw = dict(configs.CUB_TPS)
    gen = torch.Generator().manual_seed(1234)
    seed_t = torch.zeros(1, dtype=torch.int64, device="cuda")
    count = [0]

    def int_seed():
        count[0] += 1
        M.make_tps(views, kw, seed=count[0])

    def tensor_seed():
        seed_t.add_(1)
        M.make_tps(views, kw, seed=seed_t)

    return dict(generator=lambda: M.make_tps(views, kw, generator=gen), int_seed=int_seed, tensor_seed=tensor_seed)


def tiny_step_arms(torch, M, configs):
    cfg = configs.CUB_SHIPPED
    B, S, K, F = cfg.batch_size, cfg.spatial_size, cfg.n_parts, cfg.local_app_size
    torch.manual_seed(0)
    e_pi = torch.nn.Conv2d(3, K, 3, padding=1).cuda()
    e_alpha = torch.nn.Conv2d(3, 8, 3, padding=1).cuda()
    lin = torch.nn.Linear(8, F).cuda()
    dd = torch.nn.Conv2d(F + K, 3, 3, padding=1).cuda()
    params = [p for m in (e_pi, e_alpha, lin, dd) for p in m.parameters()]
    g = torch.Generator(device="cuda").manual_seed(1)
    views = [torch.rand(B, S, S, 3, device="cuda", generator=g) * 2 - 1 for _ in range(3)]
    seed_t = torch.zeros(1, dtype=torch.int64, device="cuda")
    nchw, nhwc = (lambda x: x.permute(0, 3, 1, 2)), (lambda x: x.permute(0, 2, 3, 1).contiguous())

    def step():
        v0, v1, v0t = M.make_tps(views, cfg.tps_parameters, seed=seed_t)
        l0, l1 = nhwc(e_pi(nchw(v0))), nhwc(e_pi(nchw(v1)))
        m1, parts, pooled = M.part_encode(l1, v1, seed_t)
        feat = lin(torch.relu(e_alpha(nchw(parts))).mean(dim=(2, 3))).view(K, B, F).transpose(0, 1).contiguous()
        m0, labels0, inj = M.part_decode(l0, feat, seed_t)
        loss = (nhwc(dd(nchw(inj))) - v0t).square().mean() + M.categorical_kl(m0) + M.categorical_kl(m1)
        loss.backward()

    def eager():
        seed_t.add_(1)
        for p in params:
            p.grad = None
        step()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            eager()
    torch.cuda.current_stream().wait_stream(side)
    for p in params:
        p.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()

    def replay():
        seed_t.add_(1)
        graph.replay()

    return dict(eager=eager, graph=replay)


def partstep_arms(torch, configs):
    from ups_b200 import tps
    from ups_b200.step import PartStep
    B, S, K, F = 256, 128, 16, 64
    g = torch.Generator(device="cuda").manual_seed(2)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)  # noqa: E731
    views = torch.rand(3, B, S, S, 3, device="cuda", generator=g) * 2 - 1
    l0, l1, feat = r(B, S, S, K), r(B, S, S, K), r(B, K, F)
    cot = (r(B, S, S, F + K), r(K * B, S, S, 3), r(B, K, 3), r(B, S, S, K), r(B, S, S, K))
    prm = tps.tps_parameters(2 * B, seed=99, views=2, **configs.CUB_TPS)
    coord, tv = tps.make_input_tps_param(prm)
    step = PartStep(B, S, K, F, n_views=3)
    count = [0]

    def given():
        step.forward(views, coord, tv, l0, l1, feat)
        step.backward(*cot)

    def seeded():
        count[0] += 1
        step.forward(views, None, None, l0, l1, feat, tps_seed=count[0])
        step.backward(*cot)

    return dict(given_coord=given, tps_seed=seeded)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_tps_draw.py measures on the GPU; there is no CPU path"
    import ups_b200
    from ups_b200 import configs
    from ups_b200 import model as M
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    doc = dict(card=card(), torch=torch.__version__, cudnn=torch.backends.cudnn.version(), lib=ups_b200._cabi.version(),
               rounds=a.rounds, steps=a.steps)
    doc["make_tps_cub_b256_v3"] = run_arms(torch, make_tps_arms(torch, M, configs), a.rounds, a.steps, a.warmup)
    doc["tiny_step_cub_shipped"] = run_arms(torch, tiny_step_arms(torch, M, configs), a.rounds, a.steps, a.warmup)
    doc["partstep_cub_b256_k16"] = run_arms(torch, partstep_arms(torch, configs), a.rounds, a.steps, a.warmup)
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
