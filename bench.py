#!/usr/bin/env python
"""Headline benchmark: GPT-2 training throughput (tokens/s, whole job) — BASELINE.json's metric.

    python bench.py [--gpus N --steps K --warmup W] [--mode ddp|zero1|zero2|zero3] [--model small|medium|large|xl]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference from baseline/_ref, same metric/config

Workload = the reference's own (example/ddp/train.py:22-29): one fixed synthetic (1, 1024) token batch per rank,
random-init GPT-2 (small by default), AdamW lr 1e-5 wd 0.1, gradients summed across ranks; bf16 compute.
Weak scaling: per-GPU work is fixed.  Timing: W warm-up steps, then exactly K steps between
barrier+synchronize pairs, CUDA events on the launching stream, max over ranks.  The step's working set
(parameters + gradients + fp32 optimizer state, ~2.9 GB for small) is >20x the 126 MB L2, so no explicit L2 flush.

The ONE JSON line carries the headline config (`value`, ddp / GPT-2 small unless --mode/--model say otherwise) and, with the
default `--modes auto`, a `modes` block with the other BASELINE.json configs measured the same way in the same process
(zero1 / GPT-2 medium, zero2 / large, zero3 / XL: tokens/s, ms/step, peak HBM, exposed communication) — both arms emit it,
so every reference-vs-ours row comes from the same box and the same launch.  At N > 1 our arm also emits `comm_check`:
our NVLS all-reduce / reduce-to-owner / broadcast kernels against NCCL on 3 KB / 2.4 MB / 77 MB buffers, and a bitwise
comparison of the replicas' parameters after the timed steps.

`--dump-outputs DIR` (our arm) writes what the headline config's last timed step produced, as float32 `.npy` files: `loss`,
and for every parameter `param.<name>` (the model's weights) and `master.<name>` (the fp32 master copy, bf16 runs).
Tensors above DUMP_SAMPLE elements are reduced to a fixed sample of positions seeded by the array's name, so two builds run
with the same arguments can be compared file by file; rank 0 writes.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

MODEL_DIMS = {"tiny": (2, 2, 128), "small": (12, 12, 768), "medium": (24, 16, 1024), "large": (36, 20, 1280),
              "xl": (48, 25, 1600)}
# BASELINE.json configs 3-5 (the reference's example/zero{1,2,3}/train.py at the sizes the survey names)
EXTRA_MODES = [("zero1", "medium"), ("zero2", "large"), ("zero3", "xl")]
OPTIMIZER_DESC = "AdamW lr1e-5 wd0.1 (coupled L2)"
L2_DESC = "working set (params+grads+optimizer state, GBs) >> 126 MB L2; no explicit flush"
DUMP_SAMPLE = 65536            # elements kept per dumped array
DUMP_BUDGET = 12 << 20         # elements over all dumped arrays (48 MB of float32)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="ddp", choices=["ddp", "zero1", "zero2", "zero3", "single"])
    ap.add_argument("--model", default="small", choices=["tiny", "small", "medium", "large", "xl"])
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--seq", type=int, default=1024)
    ap.add_argument("--backend", default="auto", choices=["auto", "native", "dist"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"],
                    help="parameter/compute dtype of BOTH arms; fp32 = the reference scripts' own dtype (ours: TF32 tcgen05 GEMMs)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--partition", default=None, choices=["greedy", "contiguous", "balanced"],
                    help="ownership planner (default: balanced for zero1/2, contiguous for zero3 so a layer is one fetch)")
    ap.add_argument("--modes", default="auto", choices=["auto", "none", "all"],
                    help="auto: add the zero1-medium / zero2-large / zero3-xl block when the headline is the default ddp-small")
    ap.add_argument("--mode-steps", type=int, default=10, help="timed steps of each extra config in the `modes` block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="our arm: write the loss and (sampled) parameters of the last timed step as DIR/<name>.npy (float32)")
    return ap.parse_args()


def emit(obj):
    print(json.dumps(obj), flush=True)


# ------------------------------------------------------------------------------------------------------
# clock sampling DURING the timed region (standalone: the reference arm must not import our package)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons of one GPU, sampled in a background thread.  NVML when importable (≈1 ms per
    sample, so even an 80 ms timed region gets dozens of samples), `nvidia-smi` otherwise."""

    _REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
                ("hw_power_brake_slowdown", 0x80), ("sw_power_cap", 0x4))
    SMI_FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                  "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                  "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0, period_s: float = 0.005):
        self.gpu_index, self.period_s = gpu_index, period_s
        self.sm, self.max_mhz, self.reasons, self.power = [], 0.0, set(), []
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES remaps indices: resolve through the UUID-agnostic visible list when it is numeric
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if gpu_index < len(ids) and ids[gpu_index].isdigit():
                    phys = int(ids[gpu_index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._h))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        for name, bit in self._REASONS:
            if mask & bit:
                self.reasons.add(name)
        try:
            self.power.append(n.nvmlDeviceGetPowerUsage(self._h) / 1000.0)
        except Exception:
            pass

    def _sample_smi(self):
        cmd = ["nvidia-smi", f"--query-gpu={self.SMI_FIELDS}", "--format=csv,noheader,nounits", "-i", str(self.gpu_index)]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=5).stdout.strip()
        if not out:
            return
        r = [c.strip() for c in out.splitlines()[0].split(",")]
        self.sm.append(float(r[0]))
        self.max_mhz = max(self.max_mhz, float(r[1]))
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml() if self._nvml else self._sample_smi()
            except Exception:
                pass
            self._stop.wait(self.period_s if self._nvml else max(self.period_s, 0.05))

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=10)

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz or None,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": max(self.power) if self.power else None,
                "source": "nvml" if self._nvml else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------------
# shared plumbing
# ------------------------------------------------------------------------------------------------------
def setup_dist(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29577")
    os.environ.setdefault("RANK", str(rank))
    os.environ.setdefault("WORLD_SIZE", str(world))
    dist.init_process_group(backend="nccl", init_method="env://", world_size=world, rank=rank, device_id=device)
    return rank, local, world, device


def max_over_ranks(value, device):
    import torch
    import torch.distributed as dist
    if dist.is_initialized() and dist.get_world_size() > 1:
        t = torch.tensor([value], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return float(value)


def barrier_sync(device):
    import torch
    import torch.distributed as dist
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier(device_ids=[device.index])
    torch.cuda.synchronize(device)


def _dt(args):
    import torch
    return torch.bfloat16 if args.dtype == "bf16" else torch.float32


def config_block(args, mode, model, world, B, T):
    """Identical keys and values in both arms (the driver compares them)."""
    return {"model": f"gpt2-{model}", "global_batch": B * world, "seq_len": T,
            "parallelism": f"{mode}{world}" if mode != "single" else "single",
            "optimizer": OPTIMIZER_DESC, "l2": L2_DESC}


def free_cuda():
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()


def dump_outputs(out_dir, loss, opt):
    """Write the step's loss, every non-empty parameter and its fp32 master copy (where the optimizer keeps one) as float32
    ``out_dir/<name>.npy``.  Arrays longer than the per-array share of DUMP_BUDGET (at most DUMP_SAMPLE) keep the same
    sorted sample of flat positions on every run: the sampler is seeded by the array's name.  Returns the names written."""
    import zlib
    import numpy as np
    import torch
    arrays = {"loss": loss.detach().reshape(1)}
    for name, p in opt.parameters.items():
        if p.numel():
            arrays[f"param.{name}"] = p.detach()
        master = opt.state.get(name, {}).get("master")
        if master is not None and master.numel():
            arrays[f"master.{name}"] = master
    keep = min(DUMP_SAMPLE, DUMP_BUDGET // len(arrays))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        flat = t.reshape(-1)
        if flat.numel() > keep:
            pos = np.random.default_rng(zlib.crc32(name.encode())).choice(flat.numel(), size=keep, replace=False)
            flat = flat[torch.from_numpy(np.sort(pos)).to(flat.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), flat.float().cpu().numpy())
    return list(arrays)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def build_ours(args, mode, model_name, rank, world, device):
    import torch
    from collections import OrderedDict
    import tiny_deepspeed_b200 as tds
    from tiny_deepspeed_b200.models.gpt2 import GPT2Model, gpt2_config

    cfg = gpt2_config(model_name)
    torch.manual_seed(1234)  # identical replicas; DDP also broadcasts from rank 0
    if mode in ("single",):
        model = GPT2Model(cfg).to(device=device, dtype=_dt(args))
        opt = tds.AdamW(model.named_parameters(), lr=1e-5, weight_decay=1e-1)
        return cfg, model, opt
    if mode == "ddp":
        model = GPT2Model(cfg).to(device=device, dtype=_dt(args))
        model = tds.DDP(model, backend=args.backend)
        opt = tds.DDPAdamW(model.named_parameters(), lr=1e-5, weight_decay=1e-1)
        return cfg, model, opt
    ranks_map = [f"cuda:{i}" for i in range(world)]
    with torch.device("meta"):
        meta = GPT2Model(cfg)
        parts, _ = tds.partition_tensors(OrderedDict(meta.named_parameters()), ranks_map=ranks_map,
                                         evenness_priority=0,
                                         strategy=args.partition or ("contiguous" if mode == "zero3" else "balanced"))
    W = {"zero1": tds.Zero1, "zero2": tds.Zero2, "zero3": tds.Zero3}[mode]
    O = {"zero1": tds.Zero1AdamW, "zero2": tds.Zero2AdamW, "zero3": tds.Zero3AdamW}[mode]
    if mode == "zero3":
        with torch.device("meta"):
            model = GPT2Model(cfg).to(dtype=_dt(args))
        model = W(model, parts, device=device, backend=args.backend)
    else:
        model = GPT2Model(cfg).to(device=device, dtype=_dt(args))
        model = W(model, parts, backend=args.backend)
    opt = O(model.module.named_parameters(), lr=1e-5, weight_decay=1e-1, param_part_table=parts, ranks_map=ranks_map)
    return cfg, model, opt


def measure_ours(args, mode, model_name, steps, warmup, rank, local, world, device, *, with_e2e=True, with_exposed=True,
                 keep=None, check_replicas=False, dump_dir=None):
    """One config through the public API (TrainStep).  Returns the result dict (same on every rank).  With ``dump_dir``,
    rank 0 writes the outputs of the last device-timed step there (dump_outputs)."""
    import torch
    import tiny_deepspeed_b200 as tds
    from tiny_deepspeed_b200 import ops

    free_cuda()
    cfg, model, opt = build_ours(args, mode, model_name, rank, world, device)
    B, T = args.batch, min(args.seq, cfg.block_size)
    g = torch.Generator().manual_seed(100 + rank)
    x_host = torch.randint(0, cfg.vocab_size, (B, T), generator=g).pin_memory()
    y_host = torch.randint(0, cfg.vocab_size, (B, T), generator=g).pin_memory()
    x_dev, y_dev = x_host.to(device), y_host.to(device)
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    step = tds.TrainStep(model, opt, use_graph=not args.no_graph, warmup=max(warmup - 1, 1))
    ops.reset_launches()
    for _ in range(warmup):                           # includes the eager warm-ups and the graph capture
        step(x_dev, y_dev)
    while step.use_graph and step.graph is None:      # tiny --warmup: never let the capture fall into the timed region
        step(x_dev, y_dev)
    if step.use_graph:
        step(x_dev, y_dev)                            # one untimed replay
    torch.cuda.synchronize(device)
    launches_before = ops.launches()
    per_step_launches = getattr(step, "launches_per_step", None)

    # ---- kernel/device-timed arm: inputs already resident, K steps between events ---------------------
    barrier_sync(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(gpu_index=local) as clk:
        e0.record()
        for _ in range(steps):
            loss = step(x_dev, y_dev)
        e1.record()
        torch.cuda.synchronize(device)
    barrier_sync(device)
    ms_step = max_over_ranks(e0.elapsed_time(e1), device) / steps
    final_loss = float(loss.item())
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, loss, opt)

    # ---- end-to-end arm: public API call per step, pinned-host inputs in, loss out ----------------------
    e2e_ms = None
    if with_e2e:
        barrier_sync(device)
        t0 = time.perf_counter()
        for _ in range(steps):
            loss = step(x_host, y_host)                   # H2D of this step's batch from pinned memory
            loss_host.copy_(loss, non_blocking=True)      # D2H of the step's result
            torch.cuda.current_stream(device).synchronize()
            _ = float(loss_host)
        e2e_s = time.perf_counter() - t0
        barrier_sync(device)
        e2e_ms = max_over_ranks(e2e_s * 1e3, device) / steps

    if per_step_launches is None:
        per_step_launches = (ops.launches() - launches_before) // max(2 * steps, 1) if args.no_graph else step.launches_per_step
    tokens = B * T * world
    pol = getattr(model, "policy", None)
    symm_bytes = pol.symmetric_bytes() if hasattr(pol, "symmetric_bytes") else 0
    peak = torch.cuda.max_memory_allocated(device) + symm_bytes       # symmetric (VMM) buffers bypass torch's counters
    peak = max_over_ranks(float(peak), device)

    # ---- replicas bit-identical after the timed steps?  (before the stubbed steps below, whose numerics are meaningless) ----
    replicas_ok = None
    if check_replicas and world > 1 and pol is not None and getattr(pol, "mode", "") != "zero3":
        import torch.distributed as dist
        h = torch.zeros(2, dtype=torch.int64, device=device)
        for p in model.parameters():
            if p.numel():
                v = p.data.contiguous().view(torch.int16).to(torch.int64)
                h[0] += v.sum()
                h[1] += (v * v).sum() % 1_000_003
        hs = [torch.zeros_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        replicas_ok = all(bool((x == hs[0]).all()) for x in hs)

    # ---- exposed (non-overlapped) communication: same step with every collective stubbed out (timing only) --------
    exposed_ms = None
    if with_exposed and world > 1 and hasattr(pol, "comm_stub"):
        pol.comm_stub = True
        stub = tds.TrainStep(model, opt, use_graph=not args.no_graph, warmup=2)
        for _ in range(4):
            stub(x_dev, y_dev)
        barrier_sync(device)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(steps):
            stub(x_dev, y_dev)
        s1.record()
        torch.cuda.synchronize(device)
        stub_ms = max_over_ranks(s0.elapsed_time(s1), device) / steps
        exposed_ms = max(0.0, ms_step - stub_ms)
        pol.comm_stub = False
        barrier_sync(device)
        del stub
    res = {
        "config": config_block(args, mode, model_name, world, B, T),
        "value": tokens / (ms_step * 1e-3), "ms_per_step": ms_step, "final_loss": final_loss,
        "peak_hbm_bytes": int(peak), "symmetric_bytes": int(symm_bytes), "exposed_comm_ms_per_step": exposed_ms,
        "launches_per_step": int(per_step_launches), "backend": getattr(model, "backend", "local"),
        "cuda_graph": not args.no_graph, "clocks": clk.summary(), "steps": steps, "warmup": warmup,
        "replicas_bit_identical": replicas_ok,
    }
    if e2e_ms is not None:
        res["e2e"] = {"value": tokens / (e2e_ms * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_ms,
                      "h2d_bytes_per_step": int(x_host.numel() * 8 + y_host.numel() * 8), "d2h_bytes_per_step": 4}
    if keep is not None:
        keep["model"], keep["opt"], keep["step"] = model, opt, step
    else:
        del step, model, opt
        free_cuda()
    return res


def comm_check(model, rank, world, device):
    """Driver-visible correctness of the native collectives (VERDICT r1 #7): our kernels vs NCCL on three message sizes,
    plus bit-identical replicas after the timed steps (DDP / ZeRO-1/2 keep full parameters on every rank)."""
    import torch
    import torch.distributed as dist
    pol = getattr(model, "policy", None)
    if pol is None or not getattr(pol, "is_native", False):
        return {"ok": None, "skipped": "policy is not the native backend"}
    from tiny_deepspeed_b200.parallel import symm
    out = {"ok": True, "max_err": 0.0, "cases": []}
    sizes = {"3KB": 1536, "2.4MB": 1_179_648, "77MB": 38_633_472}      # bf16 elements: LN vector / c_attn weight / wte
    buf = symm.alloc(max(sizes.values()) * 2, device, pol.group)
    flat = buf.local.view(torch.bfloat16)
    for label, n in sizes.items():
        for op in ("allreduce", "reduce_to", "broadcast"):
            gen = torch.Generator(device="cpu").manual_seed(1000 + rank)
            src = (torch.randn(n, generator=gen) * 0.5).to(torch.bfloat16).to(device)
            ref = src.clone().float()
            root = (world - 1) if op != "allreduce" else 0
            if op == "allreduce":
                dist.all_reduce(ref, op=dist.ReduceOp.SUM)
            elif op == "reduce_to":
                dist.reduce(ref, dst=root, op=dist.ReduceOp.SUM)
            else:
                dist.broadcast(ref, src=root)
            flat[:n].copy_(src)
            torch.cuda.synchronize(device)
            pol.comm.barrier()
            if op == "allreduce":
                pol.comm.allreduce(buf, 0, n, f32=False, scale=1.0, blocks=pol.comm_blocks, channel=1)
            elif op == "reduce_to":
                pol.comm.reduce_to(buf, 0, n, root, f32=False, scale=1.0, blocks=pol.comm_blocks, channel=1)
            else:
                pol.comm.broadcast(buf, 0, n * 2, root, blocks=pol.comm_blocks, channel=1)
            torch.cuda.synchronize(device)
            err = 0.0
            if op != "reduce_to" or rank == root:
                got = flat[:n].float()
                # bf16 sum of `world` terms: compare against the fp32 NCCL sum rounded to bf16, relative to its scale
                denom = float(ref.abs().max().clamp_min(1e-6))
                err = float((got - ref.to(torch.bfloat16).float()).abs().max()) / denom
            err = max_over_ranks(err, device)
            tol = 0.0 if op == "broadcast" else 2.0 ** -6     # switch-side bf16 accumulation order differs from NCCL's
            out["cases"].append({"op": op, "size": label, "rel_err": err})
            out["max_err"] = max(out["max_err"], err)
            if err > tol:
                out["ok"] = False
    del flat, buf
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    os.environ.setdefault("TDS_COMM_TIMEOUT_S", "120")    # a stuck collective must fail this run, not stall it for 10 minutes
    rank, local, world, device = setup_dist(args)
    keep = {}
    head = measure_ours(args, args.mode, args.model, args.steps, args.warmup, rank, local, world, device, keep=keep,
                        check_replicas=True, dump_dir=args.dump_outputs)
    check = None
    if world > 1:
        try:
            check = comm_check(keep["model"], rank, world, device)
            if head.get("replicas_bit_identical") is not None and check.get("ok") is not None:
                check["replicas_bit_identical"] = head["replicas_bit_identical"]
                check["ok"] = bool(check["ok"] and head["replicas_bit_identical"])
        except Exception as e:  # pragma: no cover - hardware dependent
            check = {"ok": False, "error": f"{type(e).__name__}: {e}"[:300]}
    keep.clear()
    free_cuda()

    modes = None
    want_modes = args.modes == "all" or (args.modes == "auto" and args.mode == "ddp" and args.model == "small"
                                         and args.dtype == "bf16" and not args.no_graph)
    if want_modes:
        modes = {}
        for mode, model_name in EXTRA_MODES:
            key = f"{mode}-{model_name}"
            try:
                r = measure_ours(args, mode, model_name, min(args.steps, args.mode_steps), min(max(args.warmup, 3), 4),
                                 rank, local, world, device, with_e2e=False)
                modes[key] = {k: r[k] for k in ("config", "value", "ms_per_step", "final_loss", "peak_hbm_bytes",
                                               "exposed_comm_ms_per_step", "launches_per_step", "backend", "steps", "warmup")}
                modes[key]["unit"] = "tokens/s"
            except Exception as e:  # one failing extra config must not take the headline down
                import traceback
                traceback.print_exc()
                modes[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
                free_cuda()
    if rank == 0:
        out = {
            "metric": "gpt2_train_tokens_per_sec", "value": head["value"], "unit": "tokens/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic random tokens, random-init weights", "impl": "ours",
            "config": head["config"],
            "impl_details": {"backend": head["backend"], "cuda_graph": head["cuda_graph"],
                             "master_weights": "fp32 master + fp32 moments (bf16 params)"},
            "clocks": head["clocks"],
            "e2e": head.get("e2e"),
            "gpu_launches": int(head["launches_per_step"]) * args.steps,
            "launches_per_step": head["launches_per_step"],
            "final_loss": head["final_loss"], "peak_hbm_bytes": head["peak_hbm_bytes"],
            "symmetric_bytes": head["symmetric_bytes"], "exposed_comm_ms_per_step": head["exposed_comm_ms_per_step"],
        }
        if check is not None:
            out["comm_check"] = check
        if modes is not None:
            out["modes"] = modes
        emit(out)
    if dist.is_initialized():
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference package from baseline/_ref through its own public API
# ------------------------------------------------------------------------------------------------------
def measure_reference(args, mode, model_name, steps, warmup, rank, local, world, device, *, with_e2e=True):
    import torch
    from collections import OrderedDict
    from example.model import GPTConfig, GPT2Model
    import tiny_deepspeed.core as core

    free_cuda()
    L, H, C = MODEL_DIMS[model_name]
    cfg = GPTConfig(n_layer=L, n_head=H, n_embd=C)
    if model_name == "tiny":
        cfg.vocab_size, cfg.block_size = 512, 128
    torch.manual_seed(rank)  # as the reference scripts do
    B, T = args.batch, min(args.seq, cfg.block_size)
    x_host = torch.randint(0, cfg.vocab_size, (B, T)).pin_memory()
    y_host = torch.randint(0, cfg.vocab_size, (B, T)).pin_memory()
    x_dev, y_dev = x_host.to(device), y_host.to(device)
    mode = "ddp" if mode == "single" else mode
    model = GPT2Model(cfg).to(device).to(_dt(args))
    if mode == "ddp":
        model = core.DDP(model)
        opt = core.DDPAdamW(model.named_parameters(), lr=1e-5, weight_decay=1e-1)
    else:
        ranks_map = [f"cuda:{i}" for i in range(world)]
        with torch.device("meta"):
            parts, _ = core.partition_tensors(OrderedDict(GPT2Model(cfg).named_parameters()), ranks_map=ranks_map,
                                              evenness_priority=0, verbose=False)
        W = {"zero1": core.Zero1, "zero2": core.Zero2, "zero3": core.Zero3}[mode]
        O = {"zero1": core.Zero1AdamW, "zero2": core.Zero2AdamW, "zero3": core.Zero3AdamW}[mode]
        model = W(model, parts)
        opt = O(model.module.named_parameters(), lr=1e-5, weight_decay=1e-1, param_part_table=parts, ranks_map=ranks_map)

    def one_step(x, y):
        model.require_backward_grad_sync = True
        _, loss = model(x, y)
        loss.backward()
        opt.step()
        return loss

    for _ in range(warmup):
        one_step(x_dev, y_dev)
    barrier_sync(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(gpu_index=local) as clk:
        e0.record()
        for _ in range(steps):
            loss = one_step(x_dev, y_dev)
        e1.record()
        torch.cuda.synchronize(device)
    barrier_sync(device)
    ms_step = max_over_ranks(e0.elapsed_time(e1), device) / steps
    final_loss = float(loss.item())
    tokens = B * T * world
    res = {"config": config_block(args, mode, model_name, world, B, T), "value": tokens / (ms_step * 1e-3),
           "ms_per_step": ms_step, "final_loss": final_loss, "clocks": clk.summary(), "steps": steps, "warmup": warmup}
    if with_e2e:
        barrier_sync(device)
        t0 = time.perf_counter()
        for _ in range(steps):
            loss = one_step(x_host.to(device, non_blocking=True), y_host.to(device, non_blocking=True))
            _ = loss.item()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, device) / steps
        barrier_sync(device)
        res["e2e"] = {"value": tokens / (e2e_ms * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_ms,
                      "h2d_bytes_per_step": int(x_host.numel() * 16), "d2h_bytes_per_step": 4}
    res["peak_hbm_bytes"] = int(max_over_ranks(float(torch.cuda.max_memory_allocated(device)), device))
    del model, opt, loss
    free_cuda()
    return res


def run_reference(args):
    if not os.path.isdir(os.path.join(REF_DIR, "tiny_deepspeed")):
        emit({"impl": "reference", "unavailable": "baseline/_ref not installed (run baseline/install_reference.sh)"})
        return
    # nothing of ours is importable in this process: the repo root leaves sys.path and is never re-added
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != ROOT]
    sys.path.insert(0, REF_DIR)
    try:
        import torch  # noqa: F401
        import torch.distributed as dist
        import tiny_deepspeed.core as core
        assert os.path.abspath(core.__file__).startswith(REF_DIR), core.__file__
    except Exception as e:  # pragma: no cover
        emit({"impl": "reference", "unavailable": f"import failed: {type(e).__name__}: {e}"[:300]})
        return
    try:
        rank, local, world, device = setup_dist(args)
        head = measure_reference(args, args.mode, args.model, args.steps, args.warmup, rank, local, world, device)
        modes = None
        want_modes = args.modes == "all" or (args.modes == "auto" and args.mode == "ddp" and args.model == "small"
                                             and args.dtype == "bf16")
        if want_modes:
            modes = {}
            for mode, model_name in EXTRA_MODES:
                key = f"{mode}-{model_name}"
                try:
                    r = measure_reference(args, mode, model_name, min(args.steps, args.mode_steps),
                                          min(max(args.warmup, 3), 4), rank, local, world, device, with_e2e=False)
                    modes[key] = {k: r[k] for k in ("config", "value", "ms_per_step", "final_loss", "peak_hbm_bytes",
                                                   "steps", "warmup")}
                    modes[key]["unit"] = "tokens/s"
                except Exception as e:
                    import traceback
                    traceback.print_exc()
                    modes[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
                    free_cuda()
        assert "tiny_deepspeed_b200" not in sys.modules, "the reference process must never import our package"
        if rank == 0:
            out = {"metric": "gpt2_train_tokens_per_sec", "value": head["value"], "unit": "tokens/s",
                   "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
                   "data": "synthetic random tokens, random-init weights", "impl": "reference",
                   "config": head["config"],
                   "impl_details": {"note": f"unmodified reference from baseline/_ref, model.to({args.dtype}), stock standard_attention"},
                   "clocks": head["clocks"], "e2e": head.get("e2e"),
                   "final_loss": head["final_loss"], "peak_hbm_bytes": head["peak_hbm_bytes"]}
            if modes is not None:
                out["modes"] = modes
            emit(out)
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception as e:
        import traceback
        traceback.print_exc()
        if int(os.environ.get("RANK", "0")) == 0:
            emit({"impl": "reference", "unavailable": f"run failed: {type(e).__name__}: {e}"[:300]})


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        sys.path.insert(0, ROOT)
        run_ours(args)


if __name__ == "__main__":
    main()
