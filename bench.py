#!/usr/bin/env python
"""Flagship benchmark: Llama-3-8B training step (fwd + bwd + AdamW), tokens/s over the whole job.

    python bench.py --gpus N --steps K --warmup W                 # our framework (N=1 runs in-process)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                    # N > 1, one rank per GPU
    python bench.py --impl reference ...                          # the UNMODIFIED reference from baseline/_ref

Metric / config follow BASELINE.json: tokens/sec (whole box, device-timed, max over ranks), Llama-3-8B, bf16,
synthetic tokens, random-init weights, weak scaling (one 4096-token sequence per GPU per micro-step, 8 micro-steps per
optimizer step).  Parity: reference `examples/language/llama/benchmark.py`.

Parallelism (`--parallelism`, same flag and same spellings for both arms):
    tp        the configuration BASELINE.json names: TP = N + Megatron sequence parallelism over NVSwitch (`tpN+sp`)
    dp        pure data parallel with ZeRO-1 optimizer-state sharding (`zero1(dpN)`)
    both      (default) the headline `value` is the `tp` row; the `dp` row is measured in the same process with the
              same timing rules and reported under `rows` - for an 8B model on 180 GB GPUs plain data parallelism
              scales better than TP=8, and the line says so instead of hiding it.
At N = 1 the two coincide (`tp1`).  `config.parallelism` of the two arms is the same string whenever they ran the same
thing, so the driver's same-config check compares like with like.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

BASELINE_TOKENS_PER_S_8GPU = 25.83 * 4096      # BASELINE.md B1: 25.83 samples/s x 4096 tokens on 8x B200 (7B)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--model", default=os.environ.get("CB200_BENCH_MODEL", "llama3-8b"))
    p.add_argument("--seq", type=int, default=4096)
    p.add_argument("--mbs", type=int, default=1, help="sequences per GPU per step (weak scaling)")
    p.add_argument("--accum", type=int, default=int(os.environ.get("CB200_BENCH_ACCUM", "8")),
                   help="gradient accumulation micro-steps per optimizer step (the reference headline uses batch/DP 128)")
    p.add_argument("--parallelism", default=os.environ.get("CB200_BENCH_PARALLELISM", "both"),
                   choices=["tp", "dp", "both"], help="see module docstring")
    p.add_argument("--tp", type=int, default=0, help="tensor parallel size of the tp row (default: = gpus)")
    p.add_argument("--pp", type=int, default=1)
    p.add_argument("--sp-mode", default="split_gather")
    p.add_argument("--zero", type=int, default=0)
    p.add_argument("--comm-backend", default=os.environ.get("CB200_COMM_BACKEND", "auto"))
    p.add_argument("--grad-ckpt", type=float, default=float(os.environ.get("CB200_GRAD_CKPT", "0")))
    p.add_argument("--layers", type=int, default=0, help="debug only: override layer count (marks the run invalid)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--profile", default="", help="after the timed region, run ONE extra step under torch.profiler on "
                                                 "rank 0 and write the per-kernel table to this path")
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the timed steps, write what the last timed step of the headline row computed as "
                        "DIR/<name>.npy (see dump_outputs) so two builds can be compared output for output")
    return p.parse_args()


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0) -> None:
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _init_dist(args):
    import torch
    import colossalai_b200

    if "RANK" in os.environ and "WORLD_SIZE" in os.environ:
        colossalai_b200.launch_from_torch(verbose=False)
    else:
        from colossalai_b200.testing import free_port

        colossalai_b200.launch(0, 1, "127.0.0.1", free_port(), verbose=False)
    return torch.distributed.get_rank(), torch.distributed.get_world_size()


METRIC = "tokens/sec (whole job, device-timed, max over ranks) Llama-3-8B training step (fwd+bwd+AdamW)"
L2_NOTE = "working set per step (>= 2 GB weights+activations per layer) >> 126 MB L2; no explicit flush"


def row_label(kind: str, world: int, tp: int = 0, pp: int = 1, sp_mode: str = "split_gather", zero: int = 0) -> str:
    """One spelling of a parallel layout for BOTH arms (the driver compares `config.parallelism` across arms)."""
    if kind == "dp" and world > 1:
        return f"zero1(dp{world})"
    tp = tp or world
    if world == 1:
        return "tp1"
    dp = world // (tp * pp)
    return f"tp{tp}" + (f"+sp({sp_mode})" if tp > 1 else "") + (f"xpp{pp}" if pp > 1 else "") + \
        (f"xdp{dp}" if dp > 1 else "") + (f"+zero{zero}" if zero else "")


def shared_config(args, world: int, parallelism: str) -> dict:
    """The part of `config` that must read the same in both arms."""
    return {"model": args.model + (f"[layers={args.layers} DEBUG-INVALID]" if args.layers else ""),
            "global_batch": args.mbs * world * args.accum, "seq_len": args.seq, "parallelism": parallelism,
            "grad_accum": args.accum, "optimizer": "AdamW (fp32 master + moments, grad-norm clip 1.0)", "l2": L2_NOTE}


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLES_PER_TENSOR = 8192


def dump_outputs(out_dir: str, loss: float, model, optimizer) -> None:
    """Write what a training step hands back to its caller: the loss of the step (`loss.npy`, float64) and the updated
    weights (`param.<name>.npy`, float32, one file per parameter of this rank).  A weight is read from the optimizer's
    fp32 master copy where it keeps one of the parameter's shape (the bf16 working copy rounds small updates away),
    otherwise from the parameter.  Tensors larger than the per-tensor budget are sampled at fixed positions that depend
    only on the tensor's size, so equal arguments give files that can be compared element for element."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float64))
    masters = optimizer.get_working_to_master_map() or {}
    params = list(model.unwrap().named_parameters())
    per_tensor = min(DUMP_SAMPLES_PER_TENSOR, DUMP_MAX_BYTES // 4 // max(1, len(params)))
    for name, p in params:
        w = masters.get(id(p))
        w = (w if w is not None and w.shape == p.shape else p).detach().reshape(-1)
        if w.numel() > per_tensor:
            idx = torch.randint(w.numel(), (per_tensor,), generator=torch.Generator().manual_seed(0)).sort().values
            w = w[idx.to(w.device)]
        np.save(os.path.join(out_dir, f"param.{name}.npy"), w.float().cpu().numpy())


def _measure_ours(args, kind: str, rank: int, world: int, steps: int, with_e2e: bool, profile_path: str = "",
                  dump_dir: str = "") -> dict:
    """Build the model under one parallel layout through the public API (Booster + HybridParallelPlugin), time
    `steps` optimizer steps, tear everything down again."""
    import gc

    import torch
    import torch.distributed as dist

    from colossalai_b200.booster import Booster
    from colossalai_b200.booster.plugin import HybridParallelPlugin
    from colossalai_b200.kernel import launch_counter
    from colossalai_b200.lazy import LazyInitContext
    from colossalai_b200.models import build_model, get_config
    from colossalai_b200.nn.optimizer import FusedAdam
    from colossalai_b200.shardformer import GradientCheckpointConfig

    dev = torch.device("cuda", torch.cuda.current_device())
    if kind == "dp":
        tp, pp, zero = 1, 1, (1 if world > 1 else 0)
    else:
        tp, pp, zero = (args.tp or world), args.pp, args.zero
    assert world % (tp * pp) == 0
    dp = world // (tp * pp)
    cfg = get_config(args.model)
    if args.layers:
        cfg = cfg.replace(num_hidden_layers=args.layers)
    comm_backend = args.comm_backend
    if comm_backend == "auto":
        comm_backend = "nccl"
        if tp > 1:
            try:
                from colossalai_b200.parallel import fused

                comm_backend = "fused" if fused.build_available() else "nccl"
            except Exception:
                comm_backend = "nccl"
    sp_on = tp > 1 and args.sp_mode in ("split_gather", "ring")
    plugin = HybridParallelPlugin(
        tp_size=tp, pp_size=pp, precision="bf16", zero_stage=zero,
        enable_sequence_parallelism=sp_on, sequence_parallelism_mode=args.sp_mode if sp_on else None,
        enable_fused_normalization=True, enable_flash_attention=True, parallel_output=True, max_norm=1.0,
        num_microbatches=(args.mbs * args.accum if pp > 1 else None),
        gradient_checkpoint_config=GradientCheckpointConfig(args.grad_ckpt) if args.grad_ckpt > 0 else None,
        comm_backend=comm_backend)
    booster = Booster(plugin=plugin)
    torch.manual_seed(1234)
    with LazyInitContext():
        model = build_model(cfg)
    optimizer = FusedAdam(model.parameters(), lr=1e-5, betas=(0.9, 0.95), weight_decay=0.1, adamw_mode=True)
    model, optimizer, _, _, _ = booster.boost(model, optimizer)
    model.train()

    # ---- data: a TP/SP group consumes `tp * mbs` sequences per micro-step (one 4096-token sequence per GPU)
    B = args.mbs * tp
    S = args.seq
    global_batch = B * dp * args.accum
    tokens_per_step = global_batch * S
    gen = torch.Generator().manual_seed(4321 + plugin.pg_mesh.axis_rank("dp"))
    n_bufs = 4
    host_ids = [torch.randint(0, cfg.vocab_size, (args.accum, B, S), generator=gen, dtype=torch.int64).pin_memory()
                for _ in range(n_bufs)]
    dev_ids = [h.to(dev) for h in host_ids]
    h2d_bytes = host_ids[0].numel() * host_ids[0].element_size()

    def step(ids_dev) -> torch.Tensor:
        loss_acc = None
        for a in range(args.accum):
            ids = ids_dev[a]
            out = model(input_ids=ids, labels=ids, return_logits=False)
            loss = out["loss"] / args.accum
            if a == args.accum - 1:
                booster.backward(loss, optimizer)
            else:
                with booster.no_sync(model, optimizer):
                    optimizer.backward(loss)
            loss_acc = loss.detach() if loss_acc is None else loss_acc + loss.detach()
        optimizer.step()
        optimizer.zero_grad()
        return loss_acc

    def timed(n_steps: int, e2e: bool):
        dist.barrier()
        torch.cuda.synchronize()
        s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s_ev.record()
        last_loss = None
        for i in range(n_steps):
            if e2e:
                ids = host_ids[i % n_bufs].to(dev, non_blocking=True)     # pinned host -> device, every step
                last_loss = step(ids).item()                               # device -> host read of the result
            else:
                last_loss = step(dev_ids[i % n_bufs])
        e_ev.record()
        torch.cuda.synchronize()
        dist.barrier()
        ms = s_ev.elapsed_time(e_ev)
        wall = (time.perf_counter() - t0) * 1e3
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                           # max over ranks
        return t[0].item(), t[1].item(), (last_loss if not torch.is_tensor(last_loss) else last_loss.item())

    torch.cuda.reset_peak_memory_stats()
    for i in range(args.warmup):
        step(dev_ids[i % n_bufs])
    torch.cuda.synchronize()
    launch_counter.reset()
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    ms, wall_ms, loss_val = timed(steps, e2e=False)
    launches = launch_counter.count
    by_name = dict(launch_counter.by_name)
    clocks = sampler.stop() if rank == 0 else {}
    e2e = None
    last_loss = loss_val
    if with_e2e:
        ms_e, wall_e, last_loss = timed(steps, e2e=True)
        e2e = {"value": tokens_per_step * steps / (max(ms_e, wall_e) / 1e3), "unit": "tokens/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4, "ms_per_step": max(ms_e, wall_e) / steps}
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, last_loss, model, optimizer)
    value = tokens_per_step * steps / (ms / 1e3)
    fused_stats = None
    if comm_backend == "fused":
        from colossalai_b200.parallel import fused

        fused_stats = dict(fused.stats)
    row = {"parallelism": row_label(kind, world, tp, pp, args.sp_mode, zero if kind != "dp" else 0),
           "value": value, "unit": "tokens/s", "steps": steps, "ms_per_step": ms / steps,
           "wall_ms_per_step": wall_ms / steps, "global_batch": global_batch, "comm_backend": comm_backend,
           "gpu_launches": launches, "launches_by_kernel": by_name, "loss": loss_val,
           "peak_mem_mib": torch.cuda.max_memory_allocated() / 2**20, "clocks": clocks,
           "tflops_per_gpu": cfg.flops_per_token(S) * tokens_per_step / (ms / steps / 1e3) / 1e12 / world}
    if fused_stats is not None:
        row["fused_stats"] = fused_stats
    if e2e is not None:
        row["e2e"] = e2e
    if profile_path:
        _profile_one_step(step, dev_ids[0], profile_path, rank)
    # ---- tear down (a second layout may follow in this process)
    del model, optimizer, booster, plugin, dev_ids, host_ids, step, timed
    gc.collect()
    torch.cuda.empty_cache()
    return row


def run_ours(args) -> dict:
    import torch
    import torch.distributed as dist

    import colossalai_b200

    rank, world = _init_dist(args)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    kinds = {"tp": ["tp"], "dp": ["dp"], "both": ["tp", "dp"]}[args.parallelism]
    if world == 1 or (args.tp and args.tp == 1 and args.pp == 1):
        kinds = kinds[:1]                           # tp1 == dp1
    rows = []
    for i, kind in enumerate(kinds):
        # the headline row runs the K steps the driver asked for; the companion row at least 3 and half of K
        steps = args.steps if i == 0 else max(3, args.steps // 2)
        rows.append(_measure_ours(args, kind, rank, world, steps, with_e2e=not args.no_e2e,
                                  profile_path=args.profile if i == 0 else "",
                                  dump_dir=args.dump_outputs if i == 0 else ""))
    head = rows[0]
    result = {
        "metric": METRIC, "value": head["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": head["value"] / (BASELINE_TOKENS_PER_S_8GPU * world / 8.0), "dtype": "bf16",
        "data": "synthetic tokens, random-init weights", "impl": "ours",
        "config": shared_config(args, world, head["parallelism"]),
        "detail": {"comm_backend": head["comm_backend"], "grad_ckpt_ratio": args.grad_ckpt,
                   "optimizer_impl": "one-launch multi-tensor AdamW over the flat fp32 master / moment arenas",
                   "attention": os.environ.get("CB200_ATTN_BACKEND", "default"),
                   "gemm": os.environ.get("CB200_GEMM_BACKEND", "default"),
                   "baseline_note": "vs_baseline = value / (published 8xB200 7B number scaled to N GPUs)"},
        "clocks": head["clocks"], "gpu_launches": head["gpu_launches"], "launches_by_kernel": head["launches_by_kernel"],
        "loss": head["loss"], "peak_mem_mib": head["peak_mem_mib"], "wall_ms_per_step": head["wall_ms_per_step"],
        "tflops_per_gpu": head["tflops_per_gpu"],
        "rows": [{k: v for k, v in r.items() if k not in ("launches_by_kernel",)} for r in rows],
    }
    if "fused_stats" in head:
        result["fused_stats"] = head["fused_stats"]
    if "e2e" in head:
        result["e2e"] = head["e2e"]
    if rank == 0:
        print(json.dumps(result), flush=True)
    dist.barrier()
    colossalai_b200.initialize.shutdown()
    return result


def _profile_one_step(step_fn, ids, path: str, rank: int) -> None:
    """Kernel-level breakdown of one step (CUPTI through torch.profiler; never used for a reported number)."""
    import torch
    import torch.distributed as dist
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    dist.barrier()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step_fn(ids)
        torch.cuda.synchronize()
    if rank != 0:
        return
    rows = []
    for e in prof.key_averages():
        if "cuda" not in str(getattr(e, "device_type", "")).lower():
            continue
        us = float(getattr(e, "self_device_time_total", 0.0) or getattr(e, "device_time_total", 0.0) or 0.0)
        if us > 0:
            rows.append((us, int(e.count), str(e.key)))
    total = sum(r[0] for r in rows)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        f.write(f"# one training step, rank 0, sum of kernel device time = {total / 1e3:.2f} ms\n")
        f.write("# ms_total  count  pct  kernel\n")
        for us, n, name in sorted(rows, key=lambda r: -r[0])[:90]:
            f.write(f"{us / 1e3:9.3f} {n:6d} {100 * us / max(total, 1e-9):5.1f}%  {name[:170]}\n")


def run_reference(args) -> None:
    from baseline.reference_arm import run_reference_arm

    run_reference_arm(args)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
