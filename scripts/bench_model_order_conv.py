"""The step's two sides with their first convolutions folded in (N4), as autograd ops in the reference model's order
(model.encode_conv2d / model.decode_conv2d).

  (1) CUB B=256 S=128 F=64, first layers Ce = Co = 32, K=16 and K=25, without noise and with a device noise seed,
      forward + backward, alternated round by round:
        ops        encode_conv2d + decode_conv2d with autograd (fresh outputs from the caching allocator);
        partstep   PartStep(first_conv=32, encoder_conv=32): the same kernels on persistent buffers, no autograd;
        unfolded   part_encode / part_decode followed by cuDNN fp32 convolutions (TF32 off) on the part images and the
                   injected map: the model-order step without the fold.
  (2) one training step of a tiny model (e_pi / e_alpha / dd as small torch layers around the two folded ops, loss =
      reconstruction + categorical KL of m0 and m1, noise seed on the device) at CUB_SHIPPED (B=8 S=128 K=25 F=64):
      eager against one captured CUDA graph of forward, loss and backward.

Times are CUDA-event windows, median over rounds.  Prints one JSON document with the card's name and power limit (and
writes it to --out).  Usage: python scripts/bench_model_order_conv.py [--rounds 7] [--steps 10] [--out file.json]
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


def three_arms(torch, M, K, noise, rounds, steps, warmup, B=256, S=128, F=64, Co=32):
    from ups_b200.step import PartStep
    F_ = torch.nn.functional
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)  # noqa: E731
    views = torch.rand(2, B, S, S, 3, device="cuda", generator=g) * 2 - 1
    img1 = views[1]
    l0, l1, feat = r(B, S, S, K), r(B, S, S, K), r(B, K, F)
    Vd, bd, Ve, be = r(3, 3, F + K, Co) * 0.05, r(Co) * 0.1, r(3, 3, 3, Co) * 0.2, r(Co) * 0.1
    cot = dict(g_h0=r(B, S, S, Co), g_e0=r(K * B, S, S, Co), g_m0=r(B, S, S, K), g_m1=r(B, S, S, K))
    seed = torch.zeros(1, dtype=torch.int64, device="cuda") if noise else None
    step = PartStep(B, S, K, F, n_views=2, use_tps=False, first_conv=Co, encoder_conv=Co)
    step.forward_warp(views, None, None)
    leaves = [t.clone().requires_grad_() for t in (l0, l1, feat, Vd, bd, Ve, be)]
    Wd, We = Vd.permute(3, 2, 0, 1).contiguous(), Ve.permute(3, 2, 0, 1).contiguous()    # HWIO -> OIHW, once
    conv_leaves = [t.clone().requires_grad_() for t in (l0, l1, feat, Wd, bd, We, be)]

    count = [0]

    def ps_step():           # PartStep takes its seed by value: a host counter, no device work
        count[0] += 1
        step.forward_parts(l0, l1, feat, Vd, bd, Ve, be, noise_seed=count[0] if noise else None)
        step.backward(cot["g_h0"], cot["g_e0"], None, cot["g_m0"], cot["g_m1"])

    def ops_step():
        if noise:
            seed.add_(1)
        a0, a1, f, vd, bb, ve, eb = leaves
        m1, _, e0 = M.encode_conv2d(a1, img1, ve, eb, seed)
        m0, _, _, h0 = M.decode_conv2d(a0, f, vd, bb, seed)
        torch.autograd.backward([h0, e0, m0, m1], [cot["g_h0"], cot["g_e0"], cot["g_m0"], cot["g_m1"]])
        for t in leaves:
            t.grad = None

    def unfolded_step():
        if noise:
            seed.add_(1)
        a0, a1, f, wd, bb, we, eb = conv_leaves
        m1, parts, _ = M.part_encode(a1, img1, seed)
        e0 = F_.conv2d(parts.permute(0, 3, 1, 2), we, eb, padding=1).permute(0, 2, 3, 1)
        m0, _, inj = M.part_decode(a0, f, seed)
        h0 = F_.conv2d(inj.permute(0, 3, 1, 2), wd, bb, padding=1).permute(0, 2, 3, 1)
        torch.autograd.backward([h0, e0, m0, m1], [cot["g_h0"], cot["g_e0"], cot["g_m0"], cot["g_m1"]])
        for t in conv_leaves:
            t.grad = None

    arms = dict(ops=ops_step, partstep=ps_step, unfolded=unfolded_step)
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(timed(torch, fn, steps))
    out = {k: dict(ms_median=median(v), ms_rounds=v) for k, v in ms.items()}
    del step
    return out


def tiny_model(torch, K, F, Ce=32, Co=32):
    from ups_b200 import model as M

    class Tiny(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.e_pi = torch.nn.Conv2d(3, K, 3, padding=1)
            self.Ve = torch.nn.Parameter(torch.randn(3, 3, 3, Ce) * 0.2)
            self.be = torch.nn.Parameter(torch.zeros(Ce))
            self.lin = torch.nn.Linear(Ce, F)
            self.Vd = torch.nn.Parameter(torch.randn(3, 3, F + K, Co) * 0.05)
            self.bd = torch.nn.Parameter(torch.zeros(Co))
            self.out = torch.nn.Conv2d(Co, 3, 3, padding=1)

        def forward(self, views, seed):
            v0, v1, v0t = views
            B = v0.shape[0]
            l0 = self.e_pi(v0.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).contiguous()
            l1 = self.e_pi(v1.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).contiguous()
            m1, _, e0 = M.encode_conv2d(l1, v1, self.Ve, self.be, seed)
            feat = self.lin(torch.relu(e0).mean(dim=(1, 2))).view(K, B, F).transpose(0, 1).contiguous()
            m0, _, _, h0 = M.decode_conv2d(l0, feat, self.Vd, self.bd, seed)
            rec = self.out(torch.relu(h0).permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
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
    return dict(config=dict(B=B, S=S, K=K, F=F, Ce=32, Co=32),
                **{k: dict(ms_median=median(v), ms_rounds=v) for k, v in ms.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_model_order_conv.py needs a CUDA device: there is nothing to measure on the CPU")
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    from ups_b200 import model as M
    res = dict(card=card(), torch=torch.__version__, cudnn=torch.backends.cudnn.version(), tf32=False)
    for K in (16, 25):
        for noise in (False, True):
            res[f"cub_b256_k{K}_{'device_seed' if noise else 'no_noise'}"] = three_arms(torch, M, K, noise, a.rounds,
                                                                                        a.steps, a.warmup)
            torch.cuda.empty_cache()
    res["cub_shipped_train_step"] = graph_vs_eager(torch, a.rounds, a.steps, a.warmup)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
