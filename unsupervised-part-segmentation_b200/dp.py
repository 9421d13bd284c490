"""Batch-sharded data-parallel wrapper of the per-step path (one process per GPU).

The path itself has no cross-sample dependency (TPS parameters, softmax, masks, pooling and
unpooling are all indexed by the sample), so ranks exchange nothing on the data path.  The
only collective of a training step is the mean of the gradients of the encoder/decoder
parameters that surround the path (the reference trains on one GPU and has none; its IMM
baseline averages tower gradients on the host, baselines/imm/imm/train/cnn_train_multi.py:
75-118).

How the collective is done here
-------------------------------
* The flat gradient buffer lives in symmetric memory (torch.distributed._symmetric_memory:
  every rank maps every other rank's buffer over NVLink and, on NVSwitch, a multicast address
  bound to all of them).  PyTorch is plumbing: allocation and the handle exchange.
* `ups_dp_allreduce` (csrc/dp_allreduce.cu) is ONE kernel per bucket: a flag barrier over peer
  memory, an in-switch reduction of the rank's slice (`multimem.ld_reduce`), the 1/world of the
  mean applied in registers, a multicast store into every rank's buffer, a second flag barrier.
  No separate scale pass, and 16 small CTAs instead of NCCL's channel CTAs, so that the kernel
  co-resides with the persistent K4 grid.  Without a multicast object the same kernel reads and
  writes the peers' buffers directly.  If symmetric memory is not available at all the wrapper
  falls back to `ncclAllReduce(SUM)` and hands the consumer the scale (`grad_scale`).
* Two buckets, launched where their producers finish (SURVEY.md 8d: the reduction overlaps K4-K6):
    main bucket — the padding that stands for the 33 M parameters of the CNNs this repo does not contain — from the top
    of backward, overlapped with K4 and K5;
    small bucket (1024 floats) — the stand-in modules' real gradients: the decoder head's (computed in front of K4) and
    the encoder tail's (needs K4's dfeat) — after K4, overlapped with K5/K6.
  The next forward (`forward`) waits for both before its first kernel; `wait_grads()` for whoever consumes them earlier.
* The stand-in gradient kernels (~25 us) run on the main stream in front of K4 / K5; the all-reduce kernels run on the
  reducer's high-priority side stream beside K4 and K5.
"""
import ctypes
import os

import torch
import torch.distributed as dist

from . import _cabi as C

TAIL_BUCKET_FLOATS = 1024     # the stand-in encoder tail's gradient (4*F floats) lives at the head of the last 1024 floats


def two_buckets(n_floats):
    """[(0, n - 1024), (n - 1024, 1024)]: main bucket (top of backward) and tail bucket (after K4)."""
    n = (int(n_floats) + 3) // 4 * 4
    assert n >= 2 * TAIL_BUCKET_FLOATS, n
    return [(0, n - TAIL_BUCKET_FLOATS), (n - TAIL_BUCKET_FLOATS, TAIL_BUCKET_FLOATS)]


def default_allreduce_ctas(world):
    """CTAs (128 threads each) of the all-reduce kernel, from the in-step measurements of profiles/r02_tuning.md."""
    return 16 if world >= 8 else 64 if world >= 4 else 128


def default_main_bucket(world):
    """8 ranks: the main bucket's all-reduce starts before K4 and runs beside K4 and K5 with 16 CTAs (1.600 vs 1.640 ms);
    2 and 4 ranks need 128 / 64 CTAs to fill the links, which slows the persistent K4 by 0.14-0.16 ms when they share its
    SMs, so there the all-reduce starts after K4, beside K5 (N=2: 1.605 vs 1.666 ms, N=4: 1.578 vs 1.605 ms).
    profiles/r02_tuning.md."""
    return "before_k4" if world >= 8 else "after_k4"


def shard_bounds(global_batch, rank, world_size):
    """Contiguous batch shard [lo, hi) of `rank`; the first (global_batch % world) ranks get one extra."""
    base, rem = divmod(int(global_batch), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def rank_seed(seed, rank):
    """Per-rank seed for the synthetic shard (rank-offset, SURVEY.md 8d configs 3-4)."""
    return int(seed) * 1000003 + int(rank)


def init_from_env(backend=None):
    """torchrun-style rendezvous (RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, rank=rank, world_size=world,
                                    device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend, rank=rank, world_size=world)
    return rank, local, world


def _split(n, parts):
    """[(offset, length)] of `parts` contiguous pieces of n floats, every piece a multiple of 4 floats."""
    out, off = [], 0
    for i in range(parts):
        end = n if i == parts - 1 else min(n, ((n * (i + 1) // parts) + 3) // 4 * 4)
        out.append((off, end - off))
        off = end
    return out


class GradAllReducer:
    """In-place mean all-reduce of the buckets of a flat fp32 gradient buffer, on a side stream.

    impl: "peer"  — ups_dp_allreduce over symmetric memory (multicast when the fabric offers it);
          "nccl"  — ncclAllReduce(SUM); the buffer then holds the SUM and `grad_scale` = 1/world
                    is the factor the consumer applies (no extra pass over HBM);
          "gloo"  — CPU tensors (tests): all_reduce + scale inline;
          "auto"  — "peer" on CUDA when symmetric memory can be set up, else "nccl" / "gloo".
    `buckets`: [(offset, n_floats)] or an int (that many equal pieces); default one bucket.
    """

    MAX_CTAS = 4 * 148      # the signal pad is sized for this many CTAs: `n_ctas` may be changed between launches

    def __init__(self, n_floats=None, device=None, buckets=None, impl="auto", n_ctas=64, flat_grads=None,
                 bucket_bytes=None, world_size=None, group=None):
        self.world = world_size if world_size is not None else (dist.get_world_size() if dist.is_initialized() else 1)
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.group = group
        self.n_ctas = int(n_ctas)
        self.grad_scale = 1.0
        self.fallback_reason = None
        self._hdl = self._sig_hdl = None
        if flat_grads is not None:      # caller-owned buffer (CPU tests, or NCCL on an ordinary CUDA tensor)
            self.flat = flat_grads
            n_floats = flat_grads.numel()
            impl = ("nccl" if flat_grads.is_cuda else "gloo") if impl == "auto" else impl
            assert impl in ("nccl", "gloo"), "a caller-owned buffer is not symmetric memory: impl must be nccl or gloo"
        else:
            device = torch.device(device if device is not None else "cuda")
            n_floats = (int(n_floats) + 3) // 4 * 4
            if device.type != "cuda":
                impl = "gloo" if impl == "auto" else impl
                self.flat = torch.zeros(n_floats, dtype=torch.float32, device=device)
            elif self.world > 1 and impl in ("auto", "peer"):
                try:
                    self._setup_symmetric(n_floats, device)
                    impl = "peer"
                except Exception as e:  # noqa: BLE001 - any failure of the optional fast path selects NCCL
                    if impl == "peer":
                        raise
                    self.fallback_reason = f"{type(e).__name__}: {e}"[:300]
                    impl = "nccl"
                    self.flat = torch.zeros(n_floats, dtype=torch.float32, device=device)
            else:
                impl = "nccl" if impl == "auto" else impl
                self.flat = torch.zeros(n_floats, dtype=torch.float32, device=device)
        self.impl = impl
        if bucket_bytes is not None and buckets is None:
            per = max(4, int(bucket_bytes) // 4 // 4 * 4)
            buckets = [(o, min(per, n_floats - o)) for o in range(0, n_floats, per)]
        if buckets is None:
            buckets = 1
        if isinstance(buckets, int):
            buckets = _split(n_floats, buckets)
        self.bounds = [(int(o), int(n)) for o, n in buckets]
        assert all(o % 4 == 0 for o, _ in self.bounds), "bucket offsets must be multiples of 4 floats"
        self.buckets = [self.flat[o:o + n] for o, n in self.bounds]
        self.cuda = self.flat.is_cuda
        self.stream = torch.cuda.Stream(device=self.flat.device, priority=-1) if self.cuda else None
        self._done = None
        if self.impl == "nccl" and self.world > 1:
            self.grad_scale = 1.0 / self.world
        self._range_tables = {}
        if self.impl == "peer":
            for o, n in self.bounds:
                assert n % 4 == 0 or o + n == n_floats, "peer buckets are multiples of 4 floats"

    def _setup_symmetric(self, n_floats, device):
        import torch.distributed._symmetric_memory as symm
        group = self.group if self.group is not None else dist.group.WORLD
        name = group.group_name
        if hasattr(symm, "enable_symm_mem_for_group"):
            try:
                symm.enable_symm_mem_for_group(name)
            except Exception:  # noqa: BLE001 - newer torch enables it implicitly
                pass
        with torch.cuda.device(device):
            buf = symm.empty(n_floats, dtype=torch.float32, device=device)
            hdl = symm.rendezvous(buf, name)
            nsig = C.lib.ups_dp_allreduce_signal_bytes(self.world, max(self.n_ctas, self.MAX_CTAS)) // 4
            sig = symm.empty(max(int(nsig), 64), dtype=torch.int32, device=device)
            sig_hdl = symm.rendezvous(sig, name)
            buf.zero_()
            sig.zero_()
            torch.cuda.synchronize(device)
        dist.barrier(group=group)       # every pad is zero before anyone's first kernel signals into it
        self.flat, self._sig = buf, sig
        self._hdl, self._sig_hdl = hdl, sig_hdl
        self._buf_ptrs = [int(p) for p in hdl.buffer_ptrs]
        self._sig_ptrs = [int(p) for p in sig_hdl.buffer_ptrs]
        use_mc = os.environ.get("UPS_DP_MULTICAST", "1") != "0"
        self._mc_ptr = int(hdl.multicast_ptr) if (use_mc and getattr(hdl, "has_multicast_support", lambda *a: True) and
                                                  int(hdl.multicast_ptr or 0)) else 0

    @property
    def transport(self):
        """What carries the gradients: 'nvls-multicast', 'nvlink-peer', 'nccl', 'gloo' or 'none'."""
        if self.world == 1:
            return "none"
        if self.impl == "peer":
            return "nvls-multicast" if self._mc_ptr else "nvlink-peer"
        return self.impl

    def _table(self, off, n):
        """Pointer tables of the sub-range [off, off+n) floats of the flat buffer (cached)."""
        key = (off, n)
        if key not in self._range_tables:
            bufs = (ctypes.c_void_p * self.world)(*[p + 4 * off for p in self._buf_ptrs])
            sigs = (ctypes.c_void_p * self.world)(*self._sig_ptrs)
            self._range_tables[key] = (bufs, sigs, (self._mc_ptr + 4 * off) if self._mc_ptr else None, (n + 3) // 4 * 4)
        return self._range_tables[key]

    def launch(self, bucket=None, after=None, part=None, n_ctas=None):
        """Enqueue the all-reduce of one bucket (default: all) on the side stream, behind everything already
        queued on the current stream (or behind the event `after`).  part = (i, n): only the i-th of n equal pieces
        of the bucket; n_ctas overrides the reducer's CTA count for this launch."""
        if self.world == 1:
            if self.cuda:   # nothing to exchange, but whatever the caller queued on the side stream is still waited for
                if after is not None:
                    self.stream.wait_event(after)
                self._done = torch.cuda.Event()
                self._done.record(self.stream)
            return
        idx = range(len(self.buckets)) if bucket is None else [bucket]
        if not self.cuda:
            for i in idx:
                dist.all_reduce(self.buckets[i], op=dist.ReduceOp.SUM, group=self.group)
                self.buckets[i].mul_(1.0 / self.world)
            return
        dev = self.flat.device
        if after is not None:
            self.stream.wait_event(after)
        else:
            self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev), torch.cuda.stream(self.stream):
            for i in idx:
                o, n = self.bounds[i]
                if part is not None:
                    pi, pn = part
                    lo = o + (n * pi // pn) // 4 * 4
                    hi = o + n if pi == pn - 1 else o + (n * (pi + 1) // pn) // 4 * 4
                    o, n = lo, hi - lo
                if self.impl == "peer":
                    bufs, sigs, mc, n4 = self._table(o, n)
                    C.call("ups_dp_allreduce", ctypes.cast(bufs, ctypes.c_void_p), mc, ctypes.cast(sigs, ctypes.c_void_p),
                           self.rank, self.world, n4, 1.0 / self.world, int(n_ctas or self.n_ctas), self.stream.cuda_stream)
                else:
                    # SUM (not AVG): NCCL's in-switch algorithms exist for sum only; the consumer applies grad_scale
                    dist.all_reduce(self.flat[o:o + n], op=dist.ReduceOp.SUM, group=self.group)
            self._done = torch.cuda.Event()
            self._done.record(self.stream)

    def wait(self):
        """Make the current stream wait for every launched reduction (no host synchronisation)."""
        if self.cuda and self._done is not None:
            torch.cuda.current_stream(self.flat.device).wait_event(self._done)
            self._done = None


class StandInModules:
    """The two tiny parameterised modules whose gradients the wrapper all-reduces (csrc/standin.cu):
    encoder tail `feat = pooled . Wlin + blin` (model.py:50-52) and decoder head, a 1x1 conv F+K -> 3 on
    concat(feat[label], one_hot(label)) (nn.unpool_features_gathered, nn.py:2469-2487).  Same seed on every rank:
    replicas of one model."""

    def __init__(self, K, F, device, seed=0):
        g = torch.Generator().manual_seed(10_007 + int(seed))
        self.K, self.F = K, F
        self.Wlin = ((torch.rand(3, F, generator=g) * 2 - 1) / 3 ** 0.5).to(device)
        self.blin = torch.zeros(F, device=device)
        self.Whead = ((torch.rand(F + K, 3, generator=g) * 2 - 1) / (F + K) ** 0.5).to(device)
        self.bhead = torch.zeros(3, device=device)
        self.n_tail = 3 * F + F
        self.n_head = (F + K) * 3 + 3


class DataParallelPartStep:
    """PartStep on this rank's shard + the overlapped mean all-reduce of the surrounding modules' gradients.

    `n_grad_params` sizes the flat gradient buffer (default 33.3 M fp32 = the reference's e_pi + e_alpha + dv + dd +
    discriminators, SURVEY.md section 2).  Its two buckets start with the stand-in modules' real gradients
    (`grads_head`, `grads_tail`); the rest is padding that stands for the CNNs this repo does not contain."""

    def __init__(self, per_gpu_batch, spatial_size, n_parts, local_app_size=64, n_views=3, use_tps=True,
                 views_grad=False, n_grad_params=33_300_000, device="cuda", decode_bwd="auto", allreduce="auto",
                 allreduce_ctas=0, seed=0, reducer=None, standin="auto", main_bucket="auto"):
        from .step import PartStep
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        # the stand-in modules exist to feed the collective: with one rank there is none and the step is the path alone
        # (SURVEY.md 8d: "no CNN or stand-in compute inside the clock"); standin=True forces them (tests)
        self.standin = (self.world > 1) if standin == "auto" else bool(standin)
        # where the main bucket's all-reduce starts: "before_k4" (beside K4 and K5) or "after_k4" (beside K5 only);
        # measured per world size in profiles/r02_tuning.md
        env = os.environ.get("UPS_DP_MAIN_AFTER_K4")
        if env is not None:
            main_bucket = "after_k4" if env == "1" else "before_k4"
        if main_bucket == "auto":
            main_bucket = default_main_bucket(self.world)
        assert main_bucket in ("before_k4", "after_k4"), main_bucket
        self.main_after_k4 = main_bucket == "after_k4"
        # experiment knob: UPS_DP_SPLIT=<ctas>: first half of the main bucket before K4, second half after K4 with <ctas> CTAs
        self.split_ctas = int(os.environ.get("UPS_DP_SPLIT", "0"))
        self.main_split = self.split_ctas > 0
        # rank r holds samples [r*B, (r+1)*B) of the global batch: with the same noise seed on every rank, the N ranks draw
        # exactly the logit noise that one GPU draws over the global batch (PartStep.forward(noise_seed=...))
        self.step = PartStep(per_gpu_batch, spatial_size, n_parts, local_app_size, n_views, use_tps, views_grad, device,
                             decode_bwd=decode_bwd, sample_offset=self.rank * int(per_gpu_batch))
        dev = self.step.device
        K, F = self.step.K, self.step.F
        self.mod = StandInModules(K, F, dev, seed)
        if reducer is None:     # `reducer`: an existing two-bucket GradAllReducer (one symmetric allocation per process)
            n = (max(int(n_grad_params), 4 * TAIL_BUCKET_FLOATS) + 3) // 4 * 4
            reducer = GradAllReducer(n, dev, buckets=two_buckets(n), impl=allreduce,
                                     n_ctas=allreduce_ctas or default_allreduce_ctas(self.world))
        assert len(reducer.bounds) == 2
        n_dec = reducer.bounds[1][0]
        self.reducer = reducer
        self.grads = self.reducer.flat
        # both stand-in gradients live in the small bucket (reduced after K4, when the tail's gradient exists); the main
        # bucket is padding only, so its all-reduce starts at the very top of backward, beside the head's gradient kernels
        self.tail_off = n_dec
        self.head_off = n_dec + (self.mod.n_tail + 3) // 4 * 4
        assert self.head_off + self.mod.n_head <= n_dec + reducer.bounds[1][1], "stand-in gradients exceed the small bucket"
        self.grads_tail = self.grads[self.tail_off:self.tail_off + self.mod.n_tail]        # [dWlin (3*F), dblin (F)]
        self.grads_head = self.grads[self.head_off:self.head_off + self.mod.n_head]        # [dWhead ((F+K)*3), dbhead (3)]
        B, P = self.step.B, self.step.P
        self._ws = torch.empty(max(int(C.lib.ups_standin_workspace_bytes(B, P, K, F)), 16), dtype=torch.uint8, device=dev)
        self._ev = torch.cuda.Event()

    # ---------------------------------------------------------------- forward
    def forward(self, views, coord, t_vector, l0, l1, feat, conv_V=None, conv_b=None, noise_seed=None, noise_level=1.0):
        """PartStep.forward on this rank's shard; pass the same noise_seed on every rank."""
        # the parameters (hence the averaged gradients of the previous step) are needed from the first kernel that consumes
        # logits or features; the 11x11 TPS solves in front of it depend on the batch's warp parameters only
        inner = self.step._inner if self.step.Kp else self.step
        if inner.fuse_fwd:
            inner.before_params = self.reducer.wait
        else:
            self.reducer.wait()
        return self.step.forward(views, coord, t_vector, l0, l1, feat, conv_V, conv_b, noise_seed=noise_seed,
                                 noise_level=noise_level)

    def wait_grads(self):
        """The current stream waits until both buckets hold the mean over ranks (times 1/grad_scale for NCCL)."""
        self.reducer.wait()

    # ---------------------------------------------------------------- backward
    def backward(self, g_inj, g_parts, g_pooled=None, g_m0=None, g_m1=None, g_warped=None, g_recon=None):
        """PartStep.backward plus the two gradient buckets.  g_recon [B,S,S,3]: cotangent of the stand-in decoder
        head's output (None: the head contributes no gradient this step; the buckets are reduced all the same)."""
        st, red, mod = self.step, self.reducer, self.mod
        dev = st.device
        B, P, K, F = st.B, st.P, st.K, st.F
        main = torch.cuda.current_stream(dev)
        # main bucket (padding for the 33 M parameters of the CNNs that are not here): reducible from the top of backward.
        after_k4 = self.main_after_k4
        split = self.main_split            # experiment knob: first half beside K4, second half beside K5
        if split:
            red.launch(0, part=(0, 2))
        elif not after_k4:
            red.launch(0)                  # side stream, behind what is queued on the main stream so far
        # the stand-in head's gradient (decoder side: exists before the path's backward).  The stand-in kernels run on
        # the MAIN stream (~35 us): on a side stream they shared the SMs with the persistent K4 grid, took ten times as
        # long and held the all-reduce behind them (profiles/r02_tuning.md)
        if g_recon is not None and self.standin:
            with torch.cuda.device(dev):
                C.call("ups_standin_head_bwd", g_recon.data_ptr(), st.labels0.data_ptr(), st._feat.data_ptr(),
                       self.grads_head.data_ptr(), B, P, K, F, self._ws.data_ptr(), self._ws.numel(), main.cuda_stream)
        if st.Kp:   # padded part count: the step's backward is one call (K4 and K5 inside)
            out = st.backward(g_inj, g_parts, g_pooled, g_m0, g_m1, g_warped)
        else:
            out = st.backward_decode(g_inj, g_m0)
        if split:
            red.launch(0, part=(1, 2), n_ctas=self.split_ctas)
        elif after_k4:
            red.launch(0)
        # tail bucket: the encoder tail's gradient needs dfeat (K4)
        if self.standin:
            with torch.cuda.device(dev):
                pooled, dfeat = st.pooled.contiguous(), st.dfeat.contiguous()     # views of row-pitched buffers for a padded K
                C.call("ups_standin_tail_bwd", pooled.data_ptr(), dfeat.data_ptr(), self.grads_tail.data_ptr(), B, K, 3, F,
                       self._ws.data_ptr(), self._ws.numel(), main.cuda_stream)
        red.launch(1)
        if st.Kp:
            return out
        out.update(st.backward_encode(g_parts, g_pooled, g_m1, g_warped))
        return out
