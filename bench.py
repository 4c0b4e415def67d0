#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on B200s: SAE training tokens/sec + run_with_cache images/sec, % of roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|sae|vit]
                    [--dtype fp32|bf16] [--batch B] [--model b32|l14] [--dump-outputs DIR]

The default invocation measures BOTH hot paths and prints ONE JSON line:

  top level    the SAE training step (cfg #3: d_model 768, dict 768 x 32, TopK k = 32, 4096 tokens per step per GPU, fp32) driven
               through the public ``VisionSAETrainer.train_step`` -- the first half of BASELINE.json's metric and the only path with
               a collective (N > 1: NVLink peer-memory reduce-scatter + sharded Adam + all-gather, no NCCL on the data path);
  "secondary"  the complete record of ``HookedViT.run_with_cache`` (cfg #2: CLIP ViT-B/32, batch 512 per GPU, all hook points) in
               the reference's default dtype (fp32: 3xTF32 tensor-core products); "secondary_bf16" the same call with a bf16 model.

Per record:
  value      whole-job throughput with inputs resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e        the same metric through the public API with HOST (pinned) inputs: H2D of the step's input + the call + D2H of the
             step's result inside the timed region
  roofline   SAE: the step's algorithmic bytes (SURVEY 8d: 80 d F + 8 Bt d) / step time against the measured HBM copy
             bandwidth, plus live CUDA-event timings of every stage; ViT: the dominant GEMM's algorithmic flops against the
             measured bf16 peak.  ``traffic`` is read from the committed ncu summary under profiles/ (null if none matches).
  cpu_baseline  the oracle port (oracle/*.py) timed on this box's host cores on a bounded sample
  dp_parity  (N > 1) after the timed region every rank re-trains the reference-made fixture tests/golden/sae_tiny_b.pt through
             ``VisionSAETrainer(p2p_group=...)`` and compares losses, TopK indices, parameters and counters with the
             single-process reference run; a mismatch makes the process exit non-zero.
``--impl reference`` times the CPU implementation (the oracle port of the reference).
``--dump-outputs DIR`` writes what every timed path returned to its caller in its last timed step as DIR/<record>.<name>.npy
(OutputDump); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import re
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vit-prisma_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

SAE_CFG = dict(d_in=768, expansion=32, k=32, batch=4096, dtype="float32")     # BASELINE.json configs[2]
SAE_CFG5 = dict(d_in=768, expansion=128, k=32, batch=4096, dtype="bfloat16")  # BASELINE.json configs[4]: dict 768x128, bf16, data parallel
POOL_BATCHES = 16                                            # synthetic activation pool = 16 steps' worth of tokens (201 MB > L2)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained"),
                "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic(kernel_regex: str, prefer: str = ""):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the first kernel matching ``kernel_regex`` in the newest
    committed ``profiles/*_ncu_summary.txt`` (tools/ncu_summary.py output; file names sort by round).  Returns (bytes, file) or
    (None, None): the roofline's ``traffic`` is never a literal typed into this file."""
    prof = os.path.join(ROOT, "profiles")
    try:
        files = sorted((f for f in os.listdir(prof) if f.endswith("_ncu_summary.txt")), reverse=True)
    except OSError:
        return None, None
    files.sort(key=lambda f: (prefer not in f) if prefer else False)
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for fn in files:
        cur, got = None, {}
        for line in open(os.path.join(prof, fn)):
            if line.startswith("== "):
                if cur and len(got) == 2:
                    return got["r"] + got["w"], "profiles/" + fn
                cur, got = (line if re.search(kernel_regex, line) else None), {}
            elif cur:
                m = re.match(r"\s+dram__bytes_(read|write)\.sum\s+([0-9.]+)\s+(\w+)", line)
                if m and m.group(3) in unit:
                    got[m.group(1)[0]] = float(m.group(2)) * unit[m.group(3)]
        if cur and len(got) == 2:
            return got["r"] + got["w"], "profiles/" + fn
    return None, None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md), through NVML in this process.

    NVML is initialised when the sampler is constructed (before the warm-up steps): starting `nvidia-smi` next to the timed
    loop costs seconds of driver initialisation that stall this process's own launches, and its first sample arrives after a
    short timed region is already over.  The polling thread sleeps between reads; only samples taken between __enter__ and
    __exit__ are reported."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index=0, period_s=0.02):
        self.rows, self.active, self.stop, self.period = [], False, False, period_s
        self.h = self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            self.h, self.nv = pynvml.nvmlDeviceGetHandleByIndex(phys), pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.h = None

    def _pump(self):
        nv = self.nv
        while not self.stop:
            if self.active:
                try:
                    try:
                        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(mask)))
                except Exception:
                    pass
            time.sleep(self.period)

    def __enter__(self):
        self.active = True
        return self

    def __exit__(self, *exc):
        self.active = False

    def close(self):
        self.stop = True

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({name for _, mask in self.rows for name, bit in self.REASONS if mask & bit})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": getattr(self, "max_mhz", None) if self.h else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml (in-process, polled during the timed region)" if self.h else "unavailable"}


def _dist():
    return int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))


def _cpu_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota
    (the GPU box shows 128 CPUs but cpu.max grants 16; 128 torch threads on 16 CPUs run 150x slower)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


class Ctx:
    """Rank bookkeeping + the barrier / max-over-ranks helpers of the timing contract."""

    def __init__(self):
        self.world, self.rank, self.local = _dist()
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)      # rendezvous, IPC-handle exchange, timing reductions

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        import torch.distributed as dist
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


class OutputDump:
    """``--dump-outputs DIR``: the arrays a timed path handed its caller in its last timed step, written as DIR/<name>.npy in
    float32 (floating point) or float64 (integers, exact).  ``add`` copies to the host at once: the next call of the same path
    rewrites the engine's and the model's output buffers in place.  An array of more than ``cap`` elements is reduced to ``cap``
    flattened entries at positions drawn from a fixed seed (the same positions in every run), so the files stay under BUDGET."""
    BUDGET = 64 << 20

    def __init__(self, root):
        self.root, self.arrays = root, {}

    def add(self, name, value, cap=1 << 20):
        if value is None:
            return
        t = torch.as_tensor(value).detach()
        if t.numel() > cap:
            pos = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[pos.to(t.device)]
        self.arrays[name] = t.to("cpu", torch.float32 if t.is_floating_point() else torch.float64).numpy()

    def write(self):
        total = sum(a.nbytes for a in self.arrays.values())
        if total > self.BUDGET:
            raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {self.BUDGET}")
        os.makedirs(self.root, exist_ok=True)
        for name, a in self.arrays.items():
            np.save(os.path.join(self.root, name + ".npy"), a)


# =====================================================================================================================
# CPU legs (the only code in this file that touches oracle/)
# =====================================================================================================================
def cpu_vit_images_per_sec(budget_s=12.0, batch=16, threads=None, cfg=None, layer=None):
    """Oracle port on the host cores; ``layer`` = the activation-store call (names_filter one resid_post + stop_at_layer)."""
    from oracle.vit_oracle import CLIP_B32, recipe_state_dict, state_dict_shapes, vit_forward_with_cache
    threads = threads or _cpu_cores()
    torch.set_num_threads(threads)
    cfg = dict(cfg or CLIP_B32)
    kw = {}
    if layer is not None:
        name = f"blocks.{layer}.hook_resid_post"
        kw = dict(names_filter=lambda n: n == name, stop_at_layer=layer + 1)
    sd = recipe_state_dict(state_dict_shapes(cfg), 1234)
    x = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        vit_forward_with_cache(sd, cfg, x, **kw)  # warm-up
        n, t0 = 0, time.perf_counter()
        while True:
            vit_forward_with_cache(sd, cfg, x, **kw)
            n += 1
            dt = time.perf_counter() - t0
            if dt >= budget_s or n >= 64:
                break
    what = f"resid_post of layer {layer}, stop_at_layer {layer + 1}" if layer is not None else "all default hook points"
    return {"value": n * batch / dt, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"{n} x run_with_cache(batch {batch}) d_model {cfg['d_model']} x {cfg['n_layers']} layers fp32, {what}, oracle/vit_oracle.py, {dt:.1f}s"}


def _cpu_sae_setup(batch):
    from oracle.sae_oracle import new_adam_state
    from vit_prisma.b200.synthetic import activation_pool, sae_init_params
    d, F = SAE_CFG["d_in"], SAE_CFG["d_in"] * SAE_CFG["expansion"]
    p0 = sae_init_params(d, F)
    p = {"W_enc": p0["W_encT"].t().contiguous(), "W_dec": p0["W_dec"], "b_enc": p0["b_enc"], "b_dec": p0["b_dec"]}
    return p, new_adam_state(p), activation_pool(batch, d)


def cpu_sae_tokens_per_sec(budget_s=12.0, threads=None, batch=1024):
    """Oracle port of the reference train_step (dense autograd-equivalent formulas) on host cores, bounded sample."""
    from oracle.sae_oracle import sae_train_step
    threads = threads or _cpu_cores()
    torch.set_num_threads(threads)
    p, state, x = _cpu_sae_setup(batch)
    k = SAE_CFG["k"]
    sae_train_step(p, state, x, k, 1e-3, 1)
    n, t0 = 0, time.perf_counter()
    while True:
        sae_train_step(p, state, x, k, 1e-3, n + 2)
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 16:
            break
    return {"value": n * batch / dt, "unit": "tokens/s", "cores": threads, "kind": "port",
            "sample": f"{n} train steps x {batch} tokens (of the 4096-token step), d=768 F=24576 k=32 fp32, oracle/sae_oracle.py, {dt:.1f}s"}


def run_reference_arm(args):
    """The reference's own CPU path (its restatement, oracle/) on this box's host
    cores, same metric / unit / workload as the product arm's headline, each step a bounded sample of that workload.  Rank 0 only."""
    world, rank, _ = _dist()
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    threads = _cpu_cores()
    torch.set_num_threads(threads)
    if args.workload in ("all", "sae", "cfg5", "sae_fwd"):      # cfg5 / sae_fwd's reference leg is the headline SAE sample (the oracle is fp32, d_sae 24576)
        from oracle.sae_oracle import sae_train_step
        batch = 1024   # bounded sample of the 4096-token step: the dense products are linear in the token count
        p, state, x = _cpu_sae_setup(batch)
        k = SAE_CFG["k"]
        for i in range(max(1, min(warm, 2))):
            sae_train_step(p, state, x, k, 1e-3, i + 1)
        t0 = time.perf_counter()
        for i in range(steps):
            sae_train_step(p, state, x, k, 1e-3, i + 3)
        dt = time.perf_counter() - t0
        v, unit = steps * batch / dt, "tokens/s"
        metric = SAE_METRIC
        config = {"workload": "sae_topk_train_step", "d_in": SAE_CFG["d_in"], "d_sae": SAE_CFG["d_in"] * SAE_CFG["expansion"], "k": k,
                  "tokens_per_step": batch, "note": "bounded sample of the 4096-token step on host cores"}
        sample = f"{steps} train steps x {batch} tokens, oracle/sae_oracle.py (CPU restatement of the reference train_step)"
    else:
        from oracle.vit_oracle import CLIP_B32, CLIP_L14, recipe_state_dict, state_dict_shapes, vit_forward_with_cache
        l14 = args.model == "l14"
        cfg = dict(CLIP_L14 if l14 else CLIP_B32)
        kw = {}
        if l14:
            name = f"blocks.{args.layer}.hook_resid_post"
            kw = dict(names_filter=lambda n: n == name, stop_at_layer=args.layer + 1)
        sd = recipe_state_dict(state_dict_shapes(cfg), 1234)
        batch = 4 if l14 else 16  # bounded sample of the batch-512 workload: per-image cost is flat in batch on CPU
        x = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(0))
        with torch.no_grad():
            for _ in range(max(1, min(warm, 2))):
                vit_forward_with_cache(sd, cfg, x, **kw)
            t0 = time.perf_counter()
            for _ in range(steps):
                vit_forward_with_cache(sd, cfg, x, **kw)
            dt = time.perf_counter() - t0
        v, unit = steps * batch / dt, "images/s"
        metric = vit_metric(l14, args.layer)
        config = {"workload": f"vit_l14_run_with_cache_resid_post_l{args.layer}" if l14 else "vit_b32_run_with_cache_all_hooks",
                  "batch_per_step": batch, "note": "bounded sample of the product arm's batch on host cores"}
        sample = f"{steps} steps x batch {batch}, oracle/vit_oracle.py (CPU restatement of the reference path)"
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": config, "cpu_baseline": {"value": v, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# =====================================================================================================================
# Path A: HookedViT.run_with_cache
# =====================================================================================================================
def vit_metric(l14, layer):
    return (f"run_with_cache images/sec (CLIP ViT-L/14, blocks.{layer}.hook_resid_post, stop_at_layer={layer + 1})" if l14
            else "run_with_cache images/sec (CLIP ViT-B/32, all hook points cached)")


def build_model(dtype, device, cfg):
    from vit_prisma.b200.synthetic import recipe_state_dict
    from vit_prisma.configs.HookedViTConfig import HookedViTConfig
    from vit_prisma.models.base_vit import HookedViT
    with contextlib.redirect_stdout(io.StringIO()):
        model = HookedViT(HookedViTConfig(**cfg, dtype=dtype))
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(recipe_state_dict(shapes, 1234))
    return model.to(device, dtype).eval()


def vit_flops_per_image(cfg, stop_at_layer=None):
    """SURVEY 8d: full depth, or L = stop_at_layer without the head term."""
    N = (cfg["image_size"] // cfg["patch_size"]) ** 2
    T = N + 1
    d, H, dh, M, L = cfg["d_model"], cfg["n_heads"], cfg["d_head"], cfg["d_mlp"], cfg["n_layers"]
    CPP = cfg["n_channels"] * cfg["patch_size"] ** 2
    head = 2 * d * cfg["n_classes"]
    if stop_at_layer is not None:
        L, head = stop_at_layer, 0
    return 2 * N * CPP * d + L * (6 * T * d * H * dh + 4 * H * T * T * dh + 2 * T * H * dh * d + 4 * T * d * M) + head


def time_dominant_gemm(model, batch, dtype, iters=10):
    """MLP-in GEMM (+bias, GELU, two hook-point outputs) at the step's shape, alone on the stream, CUDA events."""
    from vit_prisma.b200 import ops
    cfg = model.cfg
    M, K, N = batch * cfg.n_tokens, cfg.d_model, cfg.d_mlp
    mlp = model.blocks[0].mlp
    win, win_lo = mlp.packed_in()
    a = torch.randn(M, K, device="cuda", dtype=dtype)
    a_lo = ops.split_tf32(a) if dtype == torch.float32 else None
    pre = torch.empty(M, N, device="cuda", dtype=dtype)
    post = torch.empty(M, N, device="cuda", dtype=dtype)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def call():
        ops.gemm(a, win, mlp.b_in, act=cfg.activation_name, a_lo=a_lo, w_lo=win_lo, out0=pre, out1=post)
    for _ in range(3):
        call()
    times = []
    for _ in range(iters):
        flush.zero_()                      # evict L2 between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    es = 4 if dtype == torch.float32 else 2
    return {"ms": ms, "flops": 2.0 * M * N * K, "bytes": float(M * K * es + N * K * es + 2 * M * N * es), "shape": [M, N, K]}


def run_vit(args, ctx, cpu_leg=True, dump=None):
    from vit_prisma.b200 import _lib as L
    from vit_prisma.b200.synthetic import CLIP_B32, CLIP_L14
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    l14 = args.model == "l14"
    CFG = CLIP_L14 if l14 else CLIP_B32
    # cfg #4 (ViT part): exactly the call VisionActivationsStore.get_activations makes (activations_store.py:262-270)
    run_kw = dict(names_filter=[f"blocks.{args.layer}.hook_resid_post"], stop_at_layer=args.layer + 1) if l14 else {}
    model = build_model(dtype, dev, CFG)
    B = args.batch
    g = torch.Generator().manual_seed(rank)
    host = torch.randn(B, 3, 224, 224, generator=g).to(dtype).pin_memory()
    x = host.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    # ---- device-resident throughput
    clocks = ClockSampler(ctx.local)
    for _ in range(args.warmup):
        out, cache = model.run_with_cache(x, **run_kw)
        del cache
    ctx.barrier()
    n_keys = 0
    launches0 = L.get_lib().pb_launch_count()
    with clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            out, cache = model.run_with_cache(x, **run_kw)
            n_keys = len(cache)
            if dump is None or i < args.steps - 1:
                del cache
        e1.record()
        ctx.barrier()
        dev_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    clocks.close()
    launches = L.get_lib().pb_launch_count() - launches0
    route = model.last_route
    if dump is not None:
        rec_name = f"vit_{args.model}_{args.dtype}"
        dump.add(f"{rec_name}.out", out)
        for name, t in cache.items():                      # 214 hook points at B/32: a small sample of each
            dump.add(f"{rec_name}.cache.{name}", t, cap=1 << 14)
        del cache

    # ---- end to end: pinned host batch -> H2D -> run_with_cache -> D2H of the model output, every step
    # result read back every step: the model output [B, n_classes]; with stop_at_layer the output is the residual stream
    # (stays on the device for the SAE), so the class-token row of every image [B, d_model] is what crosses PCIe
    out_host = torch.empty((B, CFG["d_model"] if l14 else CFG["n_classes"]), dtype=dtype).pin_memory()
    result = (lambda o: o[:, 0, :]) if l14 else (lambda o: o)
    # (the copy of batch i+1 runs on a side stream under batch i's forward -- vit_prisma.b200.prefetch.DevicePrefetcher, the
    # loader-side helper the package ships; every step's bytes still cross PCIe inside the timed region)
    from vit_prisma.b200.prefetch import DevicePrefetcher
    loader = DevicePrefetcher(None, dev)         # built once, like a DataLoader: the timed region holds per-step work only
    for xd in loader.feed(host for _ in range(max(3, args.warmup))):
        out, cache = model.run_with_cache(xd, **run_kw)
        out_host.copy_(result(out), non_blocking=True)
        del cache
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for xd in loader.feed(host for _ in range(args.steps)):
        out, cache = model.run_with_cache(xd, **run_kw)
        out_host.copy_(result(out), non_blocking=True)
        del cache
    e1.record()
    del xd
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks(e0.elapsed_time(e1))

    if rank != 0:
        del model, x, out
        torch.cuda.empty_cache()
        return None
    peaks = _peaks()
    imgs = world * B * args.steps
    value = imgs / (dev_ms / 1e3)
    e2e = imgs / (e2e_ms / 1e3)
    kern = time_dominant_gemm(model, B, dtype)
    flops_img = vit_flops_per_image(CFG, run_kw.get("stop_at_layer"))
    cache_b_img = (CFG["d_model"] * ((CFG["image_size"] // CFG["patch_size"]) ** 2 + 1) * 4) if l14 else 38_980_176   # fp32 bytes
    fp32 = dtype == torch.float32
    # fp32 mode executes 3 tensor-core passes per algorithmic flop; the roofline counts ALGORITHMIC flops
    achieved = kern["flops"] / (kern["ms"] / 1e3) / 1e12
    traffic, traffic_src = (None, None) if l14 else ncu_traffic(r"k_gemm_tc2<float" if fp32 else r"k_gemm_tc2<__nv_bfloat16|k_gemm_tc2<bf16",
                                                                prefer="gemm_fp32" if fp32 else "gemm_bf16")
    # the tensor core runs kind::tf32 at half the kind::f16 rate: the fp32-mode denominator is bf16_peak / 2 per executed pass,
    # i.e. bf16_peak / 6 per algorithmic flop of the 3-pass product (MEASURED_PEAKS.json has no TF32 entry; derived, not measured)
    mode_peak = peaks["bf16_tflops"] / 6 if fp32 else peaks["bf16_tflops"]
    roof = {"bound": "tensor", "kernel": "k_gemm_tc2 (MLP-in GEMM + bias + GELU, hook_pre/hook_post spill)", "achieved": achieved,
            "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": traffic,
            "traffic_source": traffic_src, "traffic_unit": "B/launch (ncu dram read+write)", "algorithmic_bytes": kern["bytes"],
            "executed_tensor_tflops": achieved * (3 if fp32 else 1),
            "mode_peak": mode_peak, "mode_frac": achieved / mode_peak,
            "mode_peak_source": ("bf16_tflops / 2 (kind::tf32 runs at half the kind::f16 rate) / 3 passes -- derived from the measured bf16 peak"
                                 if fp32 else "measured bf16 burst"),
            "peak_source": peaks["source"] + " bf16 burst (kernel timed alone)", "shape_MNK": kern["shape"], "kernel_ms": kern["ms"],
            "hbm_gbs_of_kernel": kern["bytes"] / (kern["ms"] / 1e3) / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"],
            "passes": 3 if fp32 else 1,
            "step_algorithmic_tflops": flops_img * imgs / (dev_ms / 1e3) / 1e12,
            "step_mode_frac": flops_img * imgs / (dev_ms / 1e3) / 1e12 / (mode_peak if fp32 else (peaks["bf16_tflops_sustained"] or mode_peak)),
            "step_cache_write_gbs": cache_b_img * (1 if fp32 else 0.5) * imgs / (dev_ms / 1e3) / 1e9}
    cpu = None if not cpu_leg else (cpu_vit_images_per_sec(batch=4, cfg=CFG, layer=args.layer) if l14 else cpu_vit_images_per_sec())
    es = 4 if fp32 else 2
    rec = {"metric": vit_metric(l14, args.layer), "value": value, "unit": "images/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
           "config": {"workload": f"vit_l14_run_with_cache_resid_post_l{args.layer}" if l14 else "vit_b32_run_with_cache_all_hooks",
                      "model": ("CLIP ViT-L/14" if l14 else "CLIP ViT-B/32") + " geometry, seeded synthetic weights",
                      "batch_per_gpu": B, "global_batch": B * world, "hook_points_cached": n_keys, "route": route,
                      "gemm": "tcgen05 3xTF32" if fp32 else "tcgen05 bf16",
                      "cache_bytes_per_image": int(cache_b_img * es / 4), "l2": "working set (activations of one layer >> 126 MB) larger than L2",
                      "parallelism": f"dp{world} (images sharded, no collective)"},
           "clocks": clocks.summary(), "gpu_launches": int(launches),
           "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(host.numel() * host.element_size()),
                   "d2h_bytes_per_step": int(out_host.numel() * out_host.element_size()), "ms_per_step": e2e_ms / args.steps,
                   "overlap": "H2D of step i+1 on a copy stream under step i (DevicePrefetcher, depth 2)"},
           "roofline": roof, "cpu_baseline": cpu}
    del model, x, out
    torch.cuda.empty_cache()
    return rec


# =====================================================================================================================
# Path B: the SAE training step through VisionSAETrainer.train_step
# =====================================================================================================================
SAE_METRIC = "SAE training tokens/sec (TopK SAE, d_model=768, dict=768x32, k=32)"


class _PoolStore:
    """Activation store stand-in with the store's contract (``storage_buffer`` [tokens, n_layers, d_in], ``next_batch()``) over a
    device-resident synthetic pool, served in fixed windows so the timed loops do no gather work of their own."""

    def __init__(self, pool_dev, batch):
        self.storage_buffer = pool_dev.unsqueeze(1)
        self.batch, self.i = batch, 0

    def window(self, i):
        j = (i % (self.storage_buffer.shape[0] // self.batch)) * self.batch
        return self.storage_buffer[j:j + self.batch]

    def next_batch(self):
        self.i += 1
        return self.window(self.i - 1)


def sae_runner_cfg(d, expansion, k, batch, lr=1e-3, **kw):
    from vit_prisma.sae.config import VisionModelSAERunnerConfig
    base = dict(d_in=d, expansion_factor=expansion, activation_fn_str="topk", activation_fn_kwargs={"k": k}, train_batch_size=batch, lr=lr,
                lr_warm_up_steps=500, lr_scheduler_name="cosineannealingwarmup", max_grad_norm=1.0, normalize_activations="layer_norm",
                b_dec_init_method="mean", initialization_method="independent", _device="cuda", _dtype="float32", n_checkpoints=0,
                log_to_wandb=False, verbose=False, checkpoint_path="/tmp/prisma_b200_bench", hook_point_layer=9)
    base.update(kw)
    with contextlib.redirect_stdout(io.StringIO()):
        return VisionModelSAERunnerConfig(**base)


def build_sae_trainer(ctx, cfg, store, group=None, init=None):
    """VisionSAETrainer on ``store``; parameters from ``init`` (state-dict-shaped) or the seeded synthetic dictionary; for
    world > 1 the trainer's own ``enable_data_parallel_if_requested`` moves them into NVLink peer-visible buffers."""
    from vit_prisma.b200.synthetic import sae_init_params
    from vit_prisma.sae.train_sae import VisionSAETrainer
    with contextlib.redirect_stdout(io.StringIO()):
        trainer = VisionSAETrainer(cfg, model=None, dataset=None, activations_store=store, p2p_group=group)
    sae = trainer.sparse_coder
    if init is None:
        p = sae_init_params(cfg.d_in, int(cfg.d_sae), device=ctx.dev)
        init = {"W_enc": p["W_encT"].t(), "W_dec": p["W_dec"], "b_enc": p["b_enc"], "b_dec": p["b_dec"]}
    with torch.no_grad():
        wt, wd, be, bd = sae._canonical_params()
        wt.copy_(init["W_enc"].t().to(ctx.dev))
        wd.copy_(init["W_dec"].to(ctx.dev))
        be.copy_(init["b_enc"].to(ctx.dev))
        bd.copy_(init["b_dec"].to(ctx.dev))
    return trainer


def dump_train_step(dump, rec_name, out, sae):
    """VisionSAETrainer.train_step's return values and the parameters the step left in the module."""
    names = ("loss", "mse_loss", "l1_loss", "l0", "act_freq_scores", "n_forward_passes_since_fired", "n_frac_active_tokens")
    for name, value in zip(names, out):
        dump.add(f"{rec_name}.{name}", value)
    for name, t in sae.state_dict().items():
        dump.add(f"{rec_name}.{name}", t)


def run_sae(args, ctx, spec=None, dump=None):
    """``spec`` = SAE_CFG (the headline, configs[2]) or SAE_CFG5 (configs[4]: bf16 storage -- parameters, state dict and activations
    in bf16; the step engine trains fp32 masters and exports the rounded parameters every step, vit_prisma/sae/sae.py)."""
    from vit_prisma.b200 import _lib as L
    from vit_prisma.b200.synthetic import activation_pool
    spec = spec or SAE_CFG
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    d, F, k, Bt = spec["d_in"], spec["d_in"] * spec["expansion"], spec["k"], spec["batch"]
    low = spec["dtype"] != "float32"
    act_dtype = torch.bfloat16 if low else torch.float32
    cfg = sae_runner_cfg(d, spec["expansion"], k, Bt, _dtype=spec["dtype"])
    pool_host = activation_pool(Bt * POOL_BATCHES, d, seed=rank).to(act_dtype).pin_memory()        # every rank: its own token shard
    store = _PoolStore(pool_host.to(dev), Bt)
    group = None
    if world > 1:      # data parallel over NVLink peer memory: Bt tokens per GPU, one global step (csrc/p2p.cu)
        from vit_prisma.b200.p2p import P2PGroup
        group = P2PGroup(rank, world, dev)
    trainer = build_sae_trainer(ctx, cfg, store, group)
    sae = trainer.sparse_coder
    act_freq, since_fired, n_frac, optimizer, scheduler = trainer.initialize_training_variables()
    trainer.initialize_geometric_medians()               # b_dec = mean of the store's buffer (rank 0's is broadcast below)
    trainer.enable_data_parallel_if_requested()
    eng = sae.step_engine()
    if world > 1:
        from vit_prisma.b200.p2p import SaeDPEngine
        assert isinstance(eng, SaeDPEngine), "trainer did not keep the data-parallel engine"
    state = {"step": 0, "tokens": 0, "n_frac": n_frac}

    def step(layer_acts):
        out = trainer.train_step(sparse_autoencoder=sae, optimizer=optimizer, scheduler=scheduler, act_freq_scores=act_freq,
                                 n_forward_passes_since_fired=since_fired, n_frac_active_tokens=state["n_frac"], layer_acts=layer_acts,
                                 n_training_steps=state["step"], n_training_tokens=state["tokens"])
        state["step"] += 1
        state["tokens"] += Bt * world
        state["n_frac"] = out[-1]
        state["out"] = out
        return out[0]                                     # loss: 0-dim device tensor

    clocks = ClockSampler(ctx.local, period_s=0.002)
    for i in range(args.warmup):
        step(store.window(i))
    ctx.barrier()
    l0 = L.get_lib().pb_launch_count()
    with clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host = time.perf_counter()
        for i in range(args.steps):
            step(store.window(args.warmup + i))
        e1.record()
        host_enqueue_ms = 1e3 * (time.perf_counter() - t_host) / args.steps
        ctx.barrier()
        dev_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    clocks.close()
    launches = L.get_lib().pb_launch_count() - l0
    if dump is not None:
        dump_train_step(dump, "sae_train" if spec is SAE_CFG else "sae_train_cfg5", state["out"], sae)
    assert sae.step_engine() is eng, "the step engine was rebuilt during training"

    # ---- e2e: pinned host tokens -> H2D -> VisionSAETrainer.train_step -> D2H of the step's loss
    loss_host = torch.empty(1).pin_memory()
    from vit_prisma.b200.prefetch import DevicePrefetcher
    host_batches = lambda n: (pool_host[(i % POOL_BATCHES) * Bt:(i % POOL_BATCHES + 1) * Bt].unsqueeze(1) for i in range(n))  # noqa: E731
    loader = DevicePrefetcher(None, dev)
    for xin in loader.feed(host_batches(max(3, args.warmup))):
        loss_host.copy_(step(xin).reshape(1), non_blocking=True)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host = time.perf_counter()
    for xin in loader.feed(host_batches(args.steps)):
        loss_host.copy_(step(xin).reshape(1), non_blocking=True)
    e1.record()
    e2e_host_ms = 1e3 * (time.perf_counter() - t_host) / args.steps
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    final_loss = float(loss_host.item())
    # ---- per-stage device times (instrumented replays of one step's stages, warm) -> which kernel dominates.
    # Collective under data parallelism (the peer-memory phases contain barriers), so every rank runs it.
    stages = eng.time_stages(store.window(0)[:, 0, :].contiguous(), float(optimizer.param_groups[0]["lr"]), since_fired, act_freq)
    ctx.barrier()
    if rank != 0:
        return None
    peaks = _peaks()
    tokens = world * Bt * args.steps
    value = tokens / (dev_ms / 1e3)
    ms_step = dev_ms / args.steps
    step_bytes = eng.algorithmic_bytes(Bt)
    step_gbs = step_bytes / (ms_step / 1e3) / 1e9
    kernels = []
    for name, info in stages.items():
        ent = {"stage": name, "ms": info["ms"]}
        if info.get("bytes"):
            ent.update(algorithmic_bytes=info["bytes"], achieved_gbs=info["bytes"] / (info["ms"] / 1e3) / 1e9,
                       hbm_frac=info["bytes"] / (info["ms"] / 1e3) / 1e9 / peaks["hbm_gbs"])
        if info.get("flops"):
            ent.update(algorithmic_flops=info["flops"], achieved_tflops=info["flops"] / (info["ms"] / 1e3) / 1e12,
                       passes=info.get("passes", 1))
        if info.get("nvlink_bytes"):
            ent.update(nvlink_bytes=info["nvlink_bytes"], nvlink_gbs=info["nvlink_bytes"] / (info["ms"] / 1e3) / 1e9)
        if info.get("ncu") and "alone" not in name:
            t, src = ncu_traffic(info["ncu"], prefer="sae")
            ent.update(traffic=t, traffic_source=src)
        kernels.append(ent)
    kernels.sort(key=lambda e: -e["ms"])
    dom = kernels[0]
    with_ncu = [e for e in kernels if "traffic" in e]
    traffic_total = sum(e["traffic"] for e in with_ncu) if with_ncu and all(e["traffic"] is not None for e in with_ncu) else None
    roof = {"bound": "hbm", "kernel": "whole training step (SURVEY 8d: 80 d F + 8 Bt d algorithmic bytes; weights + gradients + Adam state dominate)",
            "achieved": step_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": step_gbs / peaks["hbm_gbs"],
            "traffic": traffic_total, "traffic_unit": "B/step (sum of the stages' ncu dram read+write, committed summaries under profiles/)",
            "algorithmic_bytes": step_bytes, "peak_source": peaks["source"] + " HBM copy bandwidth",
            "dominant_kernel": dom, "stages": kernels}
    cpu = cpu_sae_tokens_per_sec()
    mb = d * F * 4 / 1e6
    metric = SAE_METRIC if spec is SAE_CFG else f"SAE training tokens/sec (TopK SAE, d_model={d}, dict={d}x{spec['expansion']}, k={k}, {spec['dtype']})"
    rec = {"metric": metric, "value": value, "unit": "tokens/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "fp32" if not low else "bf16 storage (parameters, activations) / fp32 masters, moments and arithmetic",
           "data": "synthetic",
           "config": {"workload": "sae_topk_train_step" if spec is SAE_CFG else "sae_topk_train_step_cfg5", "api": "VisionSAETrainer.train_step",
                      "d_in": d, "d_sae": F, "k": k,
                      "tokens_per_step_per_gpu": Bt, "global_batch": Bt * world, "engine": type(eng).__name__,
                      "encoder": eng.describe_encoder(), "normalize_activations": "layer_norm", "max_grad_norm": 1.0,
                      "l2": f"working set (2 x {mb:.0f} MB weights + 2 x {2 * mb:.0f} MB Adam state + {2 * mb:.0f} MB gradients + "
                            f"{POOL_BATCHES * Bt * d * pool_host.element_size() / 1e6:.0f} MB activation pool) larger than L2",
                      "parallelism": f"dp{world}" + (" (reduce-scatter + sharded Adam + all-gather over NVLink, no NCCL on the data path; "
                                                      + eng.describe_exchange() + ")" if world > 1 else "")},
           "clocks": clocks.summary(), "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms,
           "final_loss": final_loss,
           **({"dp_trace_ms": eng.trace_report()} if getattr(eng, "_trace", None) else {}),
           "e2e": {"value": tokens / (e2e_ms / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": Bt * d * pool_host.element_size(), "d2h_bytes_per_step": 4,
                   "ms_per_step": e2e_ms / args.steps, "host_enqueue_ms_per_step": e2e_host_ms,
                   "overlap": "H2D of step i+1 on a copy stream under step i (DevicePrefetcher, depth 2)"},
           "roofline": roof, "cpu_baseline": cpu}
    return rec


# ---------------------------------------------------------------------------------------------------------------------
def run_sae_forward(args, ctx, expansion=64, dump=None):
    """north_star's forward-only shape: SAE encoder -> TopK -> decoder at d_model 768, dict 768 x 64, 4096 tokens per call,
    against SURVEY 8(d)'s forward bytes `4*(2*Bt*d) + 4*d*F + 4*F + 4*d*min(F, Bt*k)` (sparse outputs; no dense feature_acts).
    Every rank runs its own replica (no collective); the record reports the sum."""
    from vit_prisma.b200.sae_engine import SaeStepEngine, unit_norm_rows_
    from vit_prisma.b200.synthetic import activation_pool, sae_init_params
    d, k, Bt = SAE_CFG["d_in"], SAE_CFG["k"], SAE_CFG["batch"]
    F = d * expansion
    p = sae_init_params(d, F, device=ctx.dev)
    eng = SaeStepEngine(p["W_encT"], p["W_dec"], p["b_enc"], p["b_dec"], k=k, normalize_activations="layer_norm")
    unit_norm_rows_(eng.W_dec)
    eng.refresh_lo()
    pool = activation_pool(Bt * 8, d, seed=ctx.rank).to(ctx.dev)
    n = args.steps
    # warm-up by time, not by count: on rank 0 this record follows ~12 s of host-only work (the CPU baseline) during which the GPU
    # idles and drops its clocks; a handful of 0.7 ms calls is not enough to bring them back before the timed region starts
    t_warm, i = time.perf_counter(), 0
    while i < max(args.warmup, 3) or time.perf_counter() - t_warm < 0.4:
        eng.forward(pool[(i % 8) * Bt:(i % 8 + 1) * Bt])
        i += 1
        if i % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    warm_calls = i
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        res = eng.forward(pool[(i % 8) * Bt:(i % 8 + 1) * Bt])
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1)) / n
    if dump is not None:
        for name, t in zip(("sae_out", "idx", "val"), res):
            dump.add(f"sae_forward.{name}", t)
    fb_rows, rescored = eng.fallback_rows(), eng.rescored_per_row(Bt)

    def phase_ms(bits, reps=5):                       # one phase of the fused encode alone, warm replays
        import ctypes
        from vit_prisma.b200 import _lib as L
        lib, st = L.get_lib(), torch.cuda.current_stream().cuda_stream
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            L.check(lib.pb_sae_encode_topk_fused(ctypes.byref(eng._enc_desc(Bt, bits)), st), "pb_sae_encode_topk_fused")
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    phases = {"candidate_gemm_ms": phase_ms(1), "select_rescore_ms": phase_ms(2), "exact_path_ms": phase_ms(4)}
    if ctx.rank != 0:
        return None
    peaks = _peaks()
    fwd_bytes = 4 * (2 * Bt * d) + 4 * d * F + 4 * F + 4 * d * min(F, Bt * k)
    gbs = fwd_bytes / (ms / 1e3) / 1e9
    tf32_peak = peaks["bf16_tflops"] / 2
    return {"metric": f"SAE forward tokens/sec (encoder -> TopK -> decoder, d_model={d}, dict={d}x{expansion}, k={k})",
            "value": ctx.world * Bt / (ms / 1e3), "unit": "tokens/s", "ms_per_call": ms, "n_gpus": ctx.world, "calls": n,
            "config": {"workload": "sae_forward_north_star_shape", "api": "SaeStepEngine.forward (sparse idx / val + reconstruction)",
                       "d_in": d, "d_sae": F, "k": k, "tokens_per_call": Bt, "encoder": eng.describe_encoder()},
            "phases": phases, "exact_path_rows_last_call": fb_rows, "rescored_per_row": rescored,
            "caveat": "ms_per_call is the whole SaeStepEngine.forward call (prep + fused encode + decode + two fills); in rounds-2 runs 13/14 it "
                      "measured ~3x the sum of its phases replayed alone (1.84 vs 0.61 ms).  Not diagnosed on hardware (GPU minutes ran out); "
                      "one candidate cause -- GPU clocks still down after the host-only CPU-baseline leg -- is excluded by the 0.4 s time-based "
                      "warm-up added afterwards (the ViT records, which also follow a host-only leg, never showed it).  Read the phases for the "
                      "kernels, the call figure as an upper bound",
            "warmup_calls": warm_calls,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                         "algorithmic_bytes": fwd_bytes,
                         "note": "the candidate GEMM is one TF32 tensor-core pass (fp32-exact TopK indices against the reference need at "
                                 "least that): the call is tensor-bound, not HBM-bound",
                         "encoder_tf32_frac": 2.0 * Bt * F * d / (ms / 1e3) / 1e12 / tf32_peak,
                         "tf32_peak_tflops": tf32_peak, "tf32_peak_source": "bf16 burst peak of MEASURED_PEAKS.json / 2"}}


# ---------------------------------------------------------------------------------------------------------------------
def run_cfg4(args, ctx, dump=None):
    """BASELINE.json configs[3]: CLIP ViT-L/14 run_with_cache feeding an SAE (d_model 1024, dict 1024 x 64, TopK 32), data parallel:
    every rank runs its own VisionActivationsStore over its own synthetic image shard (names_filter = one resid_post,
    stop_at_layer = layer + 1, exactly the store's call) and trains on its own token shard through VisionSAETrainer.train_step;
    the SAE step is the NVLink data-parallel step.  A "step" = one train_step on 4096 tokens per GPU INCLUDING the store refills
    it triggers (the ViT forward dominates: 257 tokens per image)."""
    from torch.utils.data import TensorDataset
    from vit_prisma.b200.synthetic import CLIP_L14
    from vit_prisma.sae.training.activations_store import VisionActivationsStore
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    vit_dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    model = build_model(vit_dtype, dev, CLIP_L14)
    d, expansion, k, Bt, layer = 1024, 64, 32, 4096, args.layer
    cfg = sae_runner_cfg(d, expansion, k, Bt, hook_point_layer=layer, layer_subtype="hook_resid_post", context_size=257, store_batch_size=32,
                         n_batches_in_buffer=8, image_size=224, num_workers=0)
    g = torch.Generator().manual_seed(100 + rank)
    images = torch.randn(256, 3, 224, 224, generator=g).to(vit_dtype)
    with contextlib.redirect_stdout(io.StringIO()):
        store = VisionActivationsStore(cfg, model, TensorDataset(images, torch.zeros(256, dtype=torch.long)), num_workers=0)
    group = None
    if world > 1:
        from vit_prisma.b200.p2p import P2PGroup
        group = P2PGroup(rank, world, dev)
    trainer = build_sae_trainer(ctx, cfg, store, group)
    sae = trainer.sparse_coder
    act_freq, since_fired, n_frac, optimizer, scheduler = trainer.initialize_training_variables()
    trainer.initialize_geometric_medians()
    trainer.enable_data_parallel_if_requested()
    eng = sae.step_engine()
    state = {"step": 0, "n_frac": n_frac}

    def step():
        batch = store.next_batch()
        while batch.shape[0] != Bt:                       # the tail of a served half-buffer: skip (DP needs equal row counts)
            batch = store.next_batch()
        out = trainer.train_step(sparse_autoencoder=sae, optimizer=optimizer, scheduler=scheduler, act_freq_scores=act_freq,
                                 n_forward_passes_since_fired=since_fired, n_frac_active_tokens=state["n_frac"], layer_acts=batch.float(),
                                 n_training_steps=state["step"], n_training_tokens=state["step"] * Bt * world)
        state["step"] += 1
        state["n_frac"] = out[-1]
        state["out"] = out
        return out[0]

    for _ in range(args.warmup):
        step()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    if dump is not None:
        dump_train_step(dump, "cfg4_sae_train", state["out"], sae)
    if rank != 0:
        return None
    tokens = world * Bt * args.steps
    return {"metric": "SAE training tokens/sec fed by CLIP ViT-L/14 run_with_cache (cfg #4: d_model 1024, dict 1024x64, k=32)",
            "value": tokens / (ms / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": f"vit {args.dtype} / sae fp32", "data": "synthetic",
            "config": {"workload": "cfg4_vit_l14_store_feeding_sae", "api": "VisionActivationsStore.next_batch + VisionSAETrainer.train_step",
                       "hook_point": cfg.hook_point, "d_in": d, "d_sae": d * expansion, "k": k, "tokens_per_step_per_gpu": Bt,
                       "store_batch_size": 32, "n_batches_in_buffer": 8, "images_per_rank": 256, "engine": type(eng).__name__,
                       "encoder": eng.describe_encoder(),
                       "parallelism": f"dp{world}" + (" (" + eng.describe_exchange() + ")" if world > 1 else "")},
            "final_loss": float(loss)}


# ---------------------------------------------------------------------------------------------------------------------
def dp_parity_gate(ctx):
    """N > 1 only, after the timed regions: the NVLink data-parallel step, driven through VisionSAETrainer(p2p_group=...), must
    reproduce the reference's single-process training of tests/golden/sae_tiny_b.pt (fixture made by the unmodified reference):
    global mse, grad norm, bit-exact TopK indices, parameters after steps 0 / 5, dead-feature counters, and identical
    parameters on every rank.  Returns (ok, detail) on every rank."""
    import torch.distributed as dist
    from vit_prisma.b200.p2p import P2PGroup, SaeDPEngine
    from vit_prisma.sae.train_sae import FusedAdamHandle, FusedSchedule
    from vit_prisma.sae.training.get_scheduler import lr_multiplier_fn
    from tests.util import load_golden
    gold = load_golden("sae_tiny_b.pt")
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    B, d, k, F = gold["batch"], gold["d_in"], gold["k"], gold["d_sae"]
    g = torch.Generator().manual_seed(gold["data_seed"])
    data = torch.randn(B * gold["n_steps"], d, generator=g) * 2.0 + torch.randn(d, generator=g)
    if B % world or F % world:
        return True, f"skipped: batch {B} / d_sae {F} not divisible by {world}"
    per = B // world
    cfg = sae_runner_cfg(d, F // d, k, per, lr=gold["lr"], normalize_activations=gold["norm"], b_dec_init_method="zeros")
    trainer = build_sae_trainer(ctx, cfg, store=object(), group=P2PGroup(rank, world, dev), init=gold["init"])   # batches are fed by hand below
    trainer.enable_data_parallel_if_requested()
    sae = trainer.sparse_coder
    eng = sae.step_engine()
    problems = []
    if not isinstance(eng, SaeDPEngine):
        problems.append(f"step_engine() returned {type(eng).__name__}, not SaeDPEngine")
    since_fired, act_freq = torch.zeros(F, device=dev), torch.zeros(F, device=dev)
    optimizer = FusedAdamHandle(gold["lr"])
    scheduler = FusedSchedule(optimizer, gold["lr"], lr_multiplier_fn("cosineannealingwarmup", warm_up_steps=gold["warm_up_steps"],
                                                                      training_steps=gold["total_steps"], lr_end=gold["lr_end"]))
    n_frac, worst = 0, 0.0
    rel = lambda got, want: float((got.double().cpu() - want.double()).abs().max() / max(float(want.double().abs().max()), 1e-30))  # noqa: E731
    for s, rec in enumerate(gold["steps"]):
        x = data[s * B + rank * per: s * B + (rank + 1) * per].to(dev).unsqueeze(1)
        out = trainer.train_step(sparse_autoencoder=sae, optimizer=optimizer, scheduler=scheduler, act_freq_scores=act_freq,
                                 n_forward_passes_since_fired=since_fired, n_frac_active_tokens=n_frac, layer_acts=x,
                                 n_training_steps=s, n_training_tokens=s * B)
        n_frac = out[-1]
        torch.cuda.synchronize()
        if sae.step_engine() is not eng:
            problems.append(f"step {s}: the trainer rebuilt the step engine")
            eng = sae.step_engine()
        sc = eng.scalars_dict()
        mse = torch.tensor([sc["mse"]], device=dev)
        dist.all_reduce(mse)                                 # shares of the global mean add up
        if abs(mse.item() - rec["mse"]) > 1e-4 * abs(rec["mse"]):
            problems.append(f"step {s}: mse {mse.item():.6g} vs reference {rec['mse']:.6g}")
        if abs(sc["grad_norm"] - rec["grad_norm"]) > 1e-4 * rec["grad_norm"]:
            problems.append(f"step {s}: grad norm {sc['grad_norm']:.6g} vs reference {rec['grad_norm']:.6g}")
        if not torch.equal(eng.idx.cpu().long(), rec["topk_idx"][rank * per:(rank + 1) * per]):
            problems.append(f"step {s}: TopK indices differ from the reference")
        if "params_after" in rec:
            ref = rec["params_after"]
            ref_dec = ref["W_dec"] / ref["W_dec"].norm(dim=1, keepdim=True)
            sd = sae.state_dict()
            for name, got, want in (("W_dec", sd["W_dec"], ref_dec), ("W_enc", sd["W_enc"], ref["W_enc"]), ("b_enc", sd["b_enc"], ref["b_enc"]),
                                    ("b_dec", sd["b_dec"], ref["b_dec"])):
                e = rel(got, want)
                worst = max(worst, e)
                if e > 1e-4:
                    problems.append(f"step {s}: {name} rel err {e:.2e}")
    if not (torch.equal(since_fired.cpu(), gold["since_fired"]) and torch.equal(act_freq.cpu(), gold["act_freq"])):
        problems.append("dead-feature counters differ from the reference")
    # every rank must hold bit-identical parameters
    sd = sae.state_dict()
    sig = torch.stack([sd[n].double().sum() for n in ("W_enc", "W_dec", "b_enc", "b_dec")] +
                      [sd[n].double().abs().sum() for n in ("W_enc", "W_dec")]).to(dev)
    lo, hi = sig.clone(), sig.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    if not torch.equal(lo, hi):
        problems.append("parameters differ between ranks after training")
    flag = torch.tensor([0.0 if problems else 1.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if problems:
        print(f"[dp_parity rank {rank}] " + "; ".join(problems), file=sys.stderr, flush=True)
    return bool(flag.item() == 1.0), {"fixture": "tests/golden/sae_tiny_b.pt (unmodified reference, single process)", "world": world,
                                      "steps": len(gold["steps"]), "worst_param_rel_err": worst, "api": "VisionSAETrainer(p2p_group=...).train_step",
                                      "problems_rank0": problems}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "sae", "vit", "cfg4", "cfg5", "sae_fwd"],
                    help="all (default) = SAE training step as the headline record + the full run_with_cache record under 'secondary'")
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"], help="ViT model dtype (the SAE step is fp32)")
    ap.add_argument("--batch", type=int, default=512, help="ViT images per step per GPU")
    ap.add_argument("--model", default="b32", choices=["b32", "l14"], help="l14 = cfg #4: ViT-L/14 with the activation store's names_filter / stop_at_layer")
    ap.add_argument("--layer", type=int, default=22, help="hook_resid_post layer cached by --model l14")
    ap.add_argument("--vit-steps", type=int, default=None, help="steps of the secondary ViT records under --workload all (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each timed path returned in its last timed step to DIR/*.npy (at most 64 MB, see OutputDump)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    ctx = Ctx()
    dump = OutputDump(args.dump_outputs) if args.dump_outputs and ctx.rank == 0 else None
    rc = 0
    try:
        line = None
        if args.workload == "cfg4":
            line = run_cfg4(args, ctx, dump=dump)
        if args.workload == "cfg5":
            line = run_sae(args, ctx, spec=SAE_CFG5, dump=dump)
        if args.workload == "sae_fwd":
            line = run_sae_forward(args, ctx, dump=dump)
        if args.workload in ("all", "sae"):
            line = run_sae(args, ctx, dump=dump)
            if ctx.world > 1:
                ok, detail = dp_parity_gate(ctx)
                if line is not None:
                    line["dp_parity"], line["dp_parity_detail"] = ok, detail
                rc = 0 if ok else 3
            try:                                           # north_star's forward-only shape (dict 768 x 64), nested; never costs the headline
                fwd = run_sae_forward(args, ctx, dump=dump)
            except Exception as e:                         # noqa: BLE001 -- reported in the line, not swallowed
                fwd = {"error": f"{type(e).__name__}: {e}"}
            if line is not None and fwd is not None:
                line["forward_north_star"] = fwd
        if args.workload in ("all", "vit"):
            vargs = argparse.Namespace(**vars(args))
            if args.workload == "all":
                vargs.steps = args.vit_steps or args.steps
                vargs.warmup = min(args.warmup, 3)
            vit = run_vit(vargs, ctx, dump=dump)
            if args.workload == "vit":
                line = vit
            elif line is not None:
                line["secondary"] = vit
            if args.workload == "all" and args.dtype == "fp32":      # the throughput mode of the same path: bf16 operands, fp32 accumulation
                vargs.dtype = "bf16"
                vit16 = run_vit(vargs, ctx, cpu_leg=False, dump=dump)
                if line is not None and vit16 is not None:
                    vit16["cpu_baseline"] = vit["cpu_baseline"] if vit else None
                    line["secondary_bf16"] = vit16
        if dump is not None:
            dump.write()
        if ctx.rank == 0 and line is not None:
            print(json.dumps(line), flush=True)
    finally:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()
    if rc:
        sys.exit(rc)


if __name__ == "__main__":
    main()
