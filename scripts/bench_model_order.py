"""The step's two sides as autograd ops in the reference model's order (model.part_encode / model.part_decode).

  (1) ops vs PartStep, CUB B=256 S=128 F=64, K=16 and K=25, alternated round by round: forward (K2 + K3) and
      forward + backward (+ K4 + K5) through the ops (fresh outputs from the caching allocator, autograd) against the
      same kernels through PartStep (persistent buffers, no autograd).
  (2) one training step of a tiny model (e_pi / e_alpha / dd as small torch convolutions around the two ops, loss =
      reconstruction + categorical KL of m0 and m1, noise seed on the device) at CUB_SHIPPED (B=8 S=128 K=25 F=64):
      eager against one captured CUDA graph of forward, loss and backward.

Times are CUDA-event windows, median over rounds.  Prints one JSON document with the card's name and power limit (and
writes it to --out).  Usage: python scripts/bench_model_order.py [--rounds 7] [--steps 20] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys

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


def ops_vs_partstep(torch, M, K, rounds, steps, warmup, B=256, S=128, F=64):
    from ups_b200.step import PartStep
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)  # noqa: E731
    views = torch.rand(2, B, S, S, 3, device="cuda", generator=g) * 2 - 1
    l0, l1, feat = r(B, S, S, K), r(B, S, S, K), r(B, K, F)
    cot = dict(g_inj=r(B, S, S, F + K), g_parts=r(K * B, S, S, 3), g_pooled=r(B, K, 3), g_m0=r(B, S, S, K),
               g_m1=r(B, S, S, K))
    step = PartStep(B, S, K, F, n_views=2, use_tps=False)
    leaves = [t.clone().requires_grad_() for t in (l0, l1, feat)]

    def ps_fwd():
        step.forward(views, None, None, l0, l1, feat)

    def ps_step():
        ps_fwd()
        step.backward(cot["g_inj"], cot["g_parts"], cot["g_pooled"], cot["g_m0"], cot["g_m1"])

    def ops_fwd():
        with torch.no_grad():
            M.part_encode(l1, views[1])
            M.part_decode(l0, feat)

    def ops_step():
        a0, a1, f = leaves
        m1, parts, pooled = M.part_encode(a1, views[1])
        m0, _, inj = M.part_decode(a0, f)
        torch.autograd.backward([m0, inj, m1, parts, pooled],
                                [cot["g_m0"], cot["g_inj"], cot["g_m1"], cot["g_parts"], cot["g_pooled"]])
        for t in leaves:
            t.grad = None

    arms = dict(partstep_fwd=ps_fwd, ops_fwd=ops_fwd, partstep_fwd_bwd=ps_step, ops_fwd_bwd=ops_step)
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(timed(torch, fn, steps))
    return {k: dict(ms_median=median(v), ms_rounds=v) for k, v in ms.items()}


def tiny_model(torch, K, F):
    from ups_b200 import model as M

    class Tiny(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.e_pi = torch.nn.Conv2d(3, K, 3, padding=1)
            self.e_alpha = torch.nn.Conv2d(3, 8, 3, padding=1)
            self.lin = torch.nn.Linear(8, F)
            self.dd = torch.nn.Conv2d(F + K, 3, 3, padding=1)

        def forward(self, views, seed):
            v0, v1, v0t = views
            B = v0.shape[0]
            l0 = self.e_pi(v0.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).contiguous()
            l1 = self.e_pi(v1.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).contiguous()
            m1, parts, pooled = M.part_encode(l1, v1, seed)
            e = torch.relu(self.e_alpha(parts.permute(0, 3, 1, 2))).mean(dim=(2, 3))
            feat = self.lin(e).view(K, B, F).transpose(0, 1).contiguous()
            m0, labels0, inj = M.part_decode(l0, feat, seed)
            rec = self.dd(inj.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
            return (rec - v0t).square().mean() + M.categorical_kl(m0) + M.categorical_kl(m1)

    return Tiny().cuda()


def graph_vs_eager(torch, rounds, steps, warmup):
    from ups_b200 import configs
    cfg = configs.CUB_SHIPPED
    B, S, K, F = cfg.batch_size, cfg.spatial_size, cfg.n_parts, cfg.local_app_size
    g = torch.Generator(device="cuda").manual_seed(1)
    views = [torch.rand(B, S, S, 3, device="cuda", generator=g) * 2 - 1 for _ in range(3)]
    model = tiny_model(torch, K, F)
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")

    def train_step():
        model.zero_grad(set_to_none=False)
        model(views, seed).backward()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(max(warmup, 2)):
            train_step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        model(views, seed).backward()

    def replay():
        seed.add_(1)               # a new draw every step
        graph.replay()

    def eager():
        seed.add_(1)
        train_step()

    arms = dict(eager=eager, cuda_graph=replay)
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(timed(torch, fn, steps))
    return dict(config=dict(B=B, S=S, K=K, F=F), **{k: dict(ms_median=median(v), ms_rounds=v) for k, v in ms.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_model_order.py needs a CUDA device: there is nothing to measure on the CPU")
    from ups_b200 import model as M
    res = dict(card=card(), torch=torch.__version__)
    for K in (16, 25):
        res[f"cub_b256_k{K}"] = ops_vs_partstep(torch, M, K, a.rounds, a.steps, a.warmup)
    res["cub_shipped_train_step"] = graph_vs_eager(torch, a.rounds, a.steps, a.warmup)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
