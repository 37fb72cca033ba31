#!/usr/bin/env python
"""Headline benchmark: GPT-2-XL training tokens/s through the Oobleck pipeline-execution hot path.

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...   # the reference path's CPU restatement (oracle port)
    python bench.py --gpus 8 --replicas 2 --model gpt2        # BASELINE config 4: 2 replicas x 4 stages (DP all-reduce)
    python bench.py --reconfig --gpus 8 --replicas 2          # second half of the metric: kill a rank, time the recovery

Workload (BASELINE.json metric / configs[2], examples/gpt3.yaml): GPT-2-XL shape (48 x 1600 x 25 heads, T=1024,
V=50257), micro-batch 2, global batch 128 sequences (64 micro-batches) per optimizer step, 1F1B over N pipeline
stages (N = --gpus; N=1 runs all 50 stage layers on one GPU), fp32 AdamW.  Synthetic wikitext-2-shaped tokens,
seed-42 HF-style initial weights.  One "step" = pipeline.train() + DP all-reduce + optimizer step, i.e.
``OobleckEngine._train_step`` (oobleck/execution/engine.py:645-649).  Prints ONE JSON line on rank 0.

At N >= 4 the line also carries ``"reconfiguration"``: after the timed region rank 0 runs tools/reconfig_bench.py twice on
the same GPUs (2 replicas x N/2 stages, and one N-stage pipeline with peer shadows), each SIGKILLing a worker inside a
training step, and records the time from the lost-node message to the first completed step.  ``--with-reconfig 0`` /
``OOB_BENCH_RECONFIG=0`` turns it off; ``OOB_BENCH_RECONFIG_BUDGET_S`` (150) bounds each run, ``OOB_BENCH_EXTRAS_BUDGET_S``
(400) all extras of a line together (the driver allows one bench.py run 870 s).  At N = 8 a third
bounded extra follows, ``"config4_dp2_x_pp4"``: BASELINE config 4 itself (GPT-2 124M, 2 replicas x 4 stages) through this
script in a torchrun of its own (``OOB_BENCH_CONFIG4=0`` skips it).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import socket
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = {
    # examples/gpt3.yaml:9-22 (GPT-2-XL shape)
    "gpt2-xl": dict(model_args=dict(n_embd=1600, n_head=25, num_hidden_layers=48, n_positions=1024),
                    microbatch=2, global_batch=128),
    # BASELINE configs[1]: GPT-2 124M, micro-batch 4
    "gpt2": dict(model_args=dict(n_embd=768, n_head=12, num_hidden_layers=12, n_positions=1024),
                 microbatch=4, global_batch=128),
    # tiny shape for smoke runs
    "tiny": dict(model_args=dict(n_embd=128, n_head=2, num_hidden_layers=2, n_positions=128, vocab_size=1000),
                 microbatch=2, global_batch=8),
}
VOCAB = 50257


def flops_per_token(E: int, L: int, T: int, V: int) -> float:
    """SURVEY 8(d): fwd+bwd, no recompute, full T x T attention as the reference computes it."""
    return 6.0 * (12 * L * E * E + E * V) + 12.0 * L * T * E


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return {"bf16_tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops"))),
                    "hbm_gbs": float(d.get("hbm_gbs")), "source": "measured"}
        except Exception:  # noqa: BLE001
            pass
    # /opt/skills/guides/B200_PROFILING.md fallback (sustained figure: the GEMMs are timed inside a long step)
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def workload_config(model: str, cfg: dict, gpus: int, replicas: int) -> dict:
    """The workload both arms are quoted on (identical dict in both JSON lines)."""
    ma = cfg["model_args"]
    stages = gpus // replicas
    return {"workload": f"{model} 1F1B train step: {ma['num_hidden_layers'] + 2} stage layers over {stages} stage(s)"
                        f" x {replicas} replica(s), micro-batch {cfg['microbatch']}, "
                        f"{cfg['global_batch'] // cfg['microbatch']} micro-batches/step, T={ma['n_positions']}, AdamW",
            "global_batch": cfg["global_batch"], "seq_len": ma["n_positions"],
            "parallelism": (f"pp{stages}" if replicas == 1 else f"dp{replicas} x pp{stages}")}


def usable_cores() -> int:
    """Host threads the CPU arm may really use: the affinity mask, a cgroup CPU quota if one is set, at most 64 (the
    oracle's eager torch ops stop scaling long before that; 128 OpenMP threads on a shared, hyper-threaded host made
    the round-2 sample run for minutes)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, int(os.environ.get("OOB_CPU_ARM_MAX_THREADS", "64"))))


def free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm (BASELINE.md section 4): the oracle's torch layers behind the engine's own pipeline code -- P gloo processes,
# a real 1F1B step over the FULL-DEPTH model, torch.set_num_threads(cores // P) -- on a bounded sample of the workload:
# micro-batch 1 x REF_SEQ tokens, P micro-batches per step.  Nothing is extrapolated: ``value`` is the tokens the sample
# really processed divided by the wall time it really took (max over the processes).
REF_SEQ = int(os.environ.get("OOB_REF_SEQ", "256"))
# wall-clock budget of one CPU-arm run (the driver gives `bench.py --impl reference` 870 s; typical on a 16-core quota:
# 7-9 s per step, 25 steps in about 220 s): past it the run stops after the current step and reports what it timed
CPU_ARM_BUDGET_S = float(os.environ.get("OOB_CPU_ARM_BUDGET_S", "600"))


def _cpu_worker(rank, world, port, model, replicas, seq, steps, warmup, threads, depth, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.set_num_threads(threads)
    t_start = time.perf_counter()

    def note(msg):
        if rank == 0 and os.environ.get("OOB_CPU_ARM_VERBOSE", "1") == "1":
            print(f"[cpu arm +{time.perf_counter() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)
    try:
        import torch.distributed as dist

        from oobleck_b200.execution.dataloader import SyntheticTokenDataset
        from oobleck_b200.execution.engine import (JobArguments, ModelArguments, OobleckArguments, OobleckEngine,
                                                   layer_cost_model)
        from oobleck_b200.planning.pipeline_template import balanced_template
        from oracle.layer import OracleLayer
        OracleLayer.fast_init = True
        cfg = MODELS[model]
        ma = dict(cfg["model_args"])
        ma["num_hidden_layers"] = depth
        stages = world // replicas
        M = stages * replicas                      # one micro-batch per stage and replica in flight
        oargs = OobleckArguments(job=JobArguments(microbatch_size=1, global_microbatch_size=M, steps=steps),
                                 model=ModelArguments(model_name="gpt2", model_tag=model, model_args=ma))
        ds = SyntheticTokenDataset(num_samples=max(64, M * (steps + warmup + 2)), seq_len=seq,
                                   vocab_size=ma.get("vocab_size", VOCAB), pin_memory=False)
        eng = OobleckEngine(rank, world, 1, None, oargs, dataset=ds, layer_cls=OracleLayer, backend="gloo")
        eng.initialize_distributed("gloo")
        t = balanced_template(layer_cost_model(eng._model, 1), stages, 1)
        eng._pipeline_templates = [t]
        note(f"engine built ({threads} threads, depth {depth}, {seq} tokens per micro-batch)")
        eng.instantiate_pipelines(M, plan=[t] * replicas)
        note("pipelines instantiated (oracle layers materialised)")
        times = []
        for it in range(warmup + steps):
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            try:
                eng._train_step()
            except StopIteration:
                eng._pipeline.reset_iterator()
                eng._train_step()
            now = time.perf_counter()
            dt = torch.tensor([now - t0, now - t_start], dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)      # every rank sees the same two numbers
            note(f"step {it} took {float(dt[0]):.2f} s")
            if it >= warmup:
                times.append(float(dt[0]))
            # a host much slower than expected: stop while the run still fits the caller's window and report the steps
            # that were really timed (same decision on every rank: it is taken on the reduced numbers)
            if times and float(dt[1]) + 1.5 * float(dt[0]) > CPU_ARM_BUDGET_S and it < warmup + steps - 1:
                note(f"budget of {CPU_ARM_BUDGET_S:.0f} s reached after {len(times)} timed step(s): stopping early")
                break
        if rank == 0:
            q.put(("ok", times, M * seq))
        if world > 1:
            dist.barrier()
    except Exception:  # noqa: BLE001
        import traceback
        q.put(("error", traceback.format_exc(), 0))
        raise


def cpu_pipeline_sample(model: str, gpus: int, replicas: int, steps: int, warmup: int, timeout: float = 800.0):
    """``_cpu_pipeline_sample_once`` with one retry if the gloo rendezvous itself failed (the free port found for it was
    taken by another process before rank 0 bound it)."""
    try:
        return _cpu_pipeline_sample_once(model, gpus, replicas, steps, warmup, timeout)
    except RuntimeError as e:
        if not any(t in str(e) for t in ("Address already in use", "EADDRINUSE", "Connection refused")):
            raise
    return _cpu_pipeline_sample_once(model, gpus, replicas, steps, warmup, timeout)


def _cpu_pipeline_sample_once(model: str, gpus: int, replicas: int, steps: int, warmup: int, timeout: float = 800.0):
    """Spawn the P gloo processes of the CPU arm and return (seconds per step list, tokens per step, description)."""
    import torch.multiprocessing as mp
    cfg = MODELS[model]
    ma = cfg["model_args"]
    cores = usable_cores()
    P = gpus
    threads = max(1, cores // P)
    depth = ma["num_hidden_layers"]
    # host memory: module + flat copies of parameters and gradients + two Adam moments = 24 B per parameter
    E, V = ma["n_embd"], ma.get("vocab_size", VOCAB)
    need = 24.0 * (12 * depth * E * E + 2 * E * V)
    try:
        import psutil
        avail = float(psutil.virtual_memory().available)
    except Exception:  # noqa: BLE001
        avail = float("inf")
    depth_note = ""
    while need > 0.6 * avail and depth > 2:
        depth //= 2
        need = 24.0 * (12 * depth * E * E + 2 * E * V)
        depth_note = f" (host RAM {avail / 2**30:.0f} GiB: depth reduced to {depth} of {ma['num_hidden_layers']} blocks)"
    # the sample is REF_SEQ tokens per step in total: P micro-batches of REF_SEQ / P tokens, so that a step costs about
    # the same host time at every N (1F1B over P CPU stages of cores / P threads each) and K + W steps fit the run
    seq = max(16, min(REF_SEQ, ma["n_positions"]) // max(1, P // replicas))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=_cpu_worker, args=(r, P, port, model, replicas, seq, steps, warmup, threads, depth, q),
                         daemon=True) for r in range(P)]
    for p in procs:
        p.start()
    # bounded wait: a CPU sample that does not come back must never take the whole benchmark down with it
    import queue as _queue
    t0 = time.perf_counter()
    msg = None
    while msg is None:
        try:
            msg = q.get(timeout=2.0)
        except _queue.Empty:
            if time.perf_counter() - t0 > timeout:
                msg = ("error", f"CPU sample exceeded its {timeout:.0f} s budget", 0)
            elif any(p.exitcode not in (None, 0) for p in procs):
                msg = ("error", "a CPU worker died: exit codes " + str([p.exitcode for p in procs]), 0)
    status, payload, tokens = msg
    for p in procs:
        p.join(timeout=5 if status != "ok" else 120)
        if p.is_alive():
            p.terminate()
    if status != "ok":
        raise RuntimeError("CPU arm failed: " + str(payload))
    sample = (f"real 1F1B train step (pipeline.train + all-reduce + AdamW) of the oracle port over {P} gloo process(es) x "
              f"{threads} threads: full depth ({depth + 2} stage layers{depth_note}), micro-batch 1 x {seq} tokens, "
              f"{tokens // seq} micro-batches per step; nothing extrapolated")
    return payload, tokens, {"cores": threads * P, "sample": sample}


def run_reference(args, cfg):
    """CPU arm: the oracle port of the reference's per-stage fwd/bwd path on the host cores (the reference itself
    hard-codes cuda/nccl/fused AdamW and cannot be installed here -- deepspeed, accelerate, HF-fx, cppcoro, oneTBB
    are all missing; DESIGN.md).  Under torchrun only rank 0 works: it spawns its own P gloo processes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for k in list(os.environ):       # the children get their own rendezvous: nothing of torchrun's may leak into them
        if k.startswith("TORCHELASTIC") or k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT",
                                                 "LOCAL_WORLD_SIZE", "GROUP_RANK", "GROUP_WORLD_SIZE", "ROLE_RANK",
                                                 "ROLE_WORLD_SIZE", "ROLE_NAME", "OMP_NUM_THREADS",
                                                 "TORCH_NCCL_ASYNC_ERROR_HANDLING"):
            os.environ.pop(k, None)
    times, tokens, info = cpu_pipeline_sample(args.model, args.gpus, args.replicas, args.steps, args.warmup)
    sec = sum(times) / len(times)
    value = tokens / sec
    if len(times) < args.steps:
        info["sample"] += f"; stopped after {len(times)} of {args.steps} timed steps ({CPU_ARM_BUDGET_S:.0f} s budget)"
    print(json.dumps({
        "impl": "reference", "metric": "training_tokens_per_s", "value": value, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.model, cfg, args.gpus, args.replicas),
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": info["cores"], "kind": "port",
                         "sample": info["sample"]},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def cpu_baseline_sample(model: str):
    """Bounded CPU sample for the N=1 line of our arm: one warm-up + two timed steps of the same CPU pipeline, with a hard
    wall-clock budget (the GPU numbers of the line must never be lost to a slow host)."""
    budget = float(os.environ.get("OOB_CPU_BASELINE_BUDGET_S", "240"))
    try:
        times, tokens, info = cpu_pipeline_sample(model, 1, 1, steps=2, warmup=1, timeout=budget)
    except RuntimeError as e:
        return {"value": None, "unit": "tokens/s", "cores": usable_cores(), "kind": "port",
                "sample": f"not measured: {str(e)[:200]}"}
    return {"value": tokens * len(times) / sum(times), "unit": "tokens/s", "cores": info["cores"], "kind": "port",
            "sample": f"{len(times)} x ({info['sample']})"}


# ---------------------------------------------------------------------------------------------------------------
def _quiet_nccl():
    # stdout carries exactly one JSON line: keep NCCL's "NCCL version ..." banner (printed to stdout at
    # NCCL_DEBUG=VERSION and above) out of it
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"


def parity_check(args, cfg, world: int, rank: int, local_rank: int, transport_cls) -> dict:
    """Before anything is timed: the benchmarked configuration (width, heads, T, micro-batch, operand format, the same
    number of pipeline stages over the same transport) at reduced depth -- one train step of 2 micro-batches -- against
    the oracle on the host: total loss and the global L2 norm of all parameter gradients.  Raises if either is off, so a
    line that was printed carries a passed check (and makes multi-GPU parity visible in the driver's records)."""
    import torch.distributed as dist

    from oobleck_b200.execution.dataloader import OobleckSampler, SyntheticTokenDataset
    from oobleck_b200.execution.engine import JobArguments, ModelArguments, OobleckArguments, OobleckEngine
    from oobleck_b200.planning.pipeline_template import even_template
    ma = dict(cfg["model_args"])
    depth = max(2, world - 2) if world > 2 else 2
    ma["num_hidden_layers"] = depth
    T, vocab, mb, M = ma["n_positions"], ma.get("vocab_size", VOCAB), cfg["microbatch"], 2
    oargs = OobleckArguments(job=JobArguments(microbatch_size=mb, global_microbatch_size=mb * M, steps=1),
                             model=ModelArguments(model_name="gpt2", model_tag="parity", model_args=ma))
    ds = SyntheticTokenDataset(num_samples=64, seq_len=T, vocab_size=vocab)
    eng = OobleckEngine(local_rank, world, 1, None, oargs, dataset=ds, nsplit=args.nsplit, transport_cls=transport_cls,
                        templates=[even_template(depth + 2, world)])
    eng.initialize_distributed()
    eng.instantiate_pipelines(M)
    eng._pipeline.train()
    torch.cuda.synchronize()
    sq = torch.zeros(1, dtype=torch.float64, device="cuda")
    for l in eng._pipeline.execution._layers:
        sq += l.flat_grad.double().pow(2).sum()
    loss = eng._pipeline.execution.total_loss.double().reshape(1) if eng._pipeline.is_last_stage() else \
        torch.zeros(1, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(sq)
        dist.all_reduce(loss)
    got_loss, got_gn = float(loss), float(sq.sqrt())
    res = {"config": f"{args.model} width at depth {depth} blocks, {world} stage(s), {M} micro-batches of {mb} x {T}",
           "loss": got_loss, "grad_norm": got_gn}
    verdict = torch.zeros(1, device="cuda")
    if rank == 0:
        from oracle import gpt2 as og
        torch.set_num_threads(usable_cores())
        d = og.GPT2Dims(n_embd=ma["n_embd"], n_head=ma["n_head"], n_layer=depth, n_positions=T, vocab_size=vocab)
        olayers = og.build_layers(d)
        for ol, spec in zip(olayers, eng._model.layers):
            og.load_flat_(ol, spec.init_flat())
        it = iter(OobleckSampler(ds, mb, 0, [M], 0))
        ref_loss = 0.0
        for _ in range(M):
            ids = ds.input_ids[next(it)]
            x = (ids, torch.ones_like(ids), ids)
            for ol in olayers:
                x = ol(*x)
            x[0].backward()
            ref_loss += float(x[0])
        ref_gn = float(sum(og.flat_grads(ol).double().pow(2).sum() for ol in olayers).sqrt())
        res.update(oracle_loss=ref_loss, oracle_grad_norm=ref_gn,
                   loss_rel_err=abs(got_loss - ref_loss) / abs(ref_loss),
                   grad_norm_rel_err=abs(got_gn - ref_gn) / abs(ref_gn), rtol=1e-4)
        res["ok"] = bool(res["loss_rel_err"] < 1e-4 and res["grad_norm_rel_err"] < 1e-4)
        verdict[0] = 1.0 if res["ok"] else 0.0
    if world > 1:
        dist.broadcast(verdict, 0)
    del eng
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    if float(verdict) != 1.0:
        raise RuntimeError(f"parity check against the oracle failed: {res}")
    return res


def busy_intervals_ms(prof, base):
    """Union length of the [start, end] windows of every forward / backward pass of one step, on this rank."""
    iv = sorted((base.elapsed_time(a), base.elapsed_time(b)) for _, a, b in prof)
    busy, cur_s, cur_e = 0.0, None, None
    for s, e in iv:
        if cur_e is None or s > cur_e:
            if cur_e is not None:
                busy += cur_e - cur_s
            cur_s, cur_e = s, e
        else:
            cur_e = max(cur_e, e)
    if cur_e is not None:
        busy += cur_e - cur_s
    return busy


DUMP_SAMPLE = 1 << 17        # parameters kept per layer: 50 GPT-2-XL layers x 512 KiB = 25 MiB


def dump_outputs(directory: str, engine):
    """What the timed step hands its caller, as float32 / float64 .npy files: the engine's running total loss (a sum over
    every micro-batch since the engine started; the engine never resets it) on the last stage, and for every layer a
    fixed sample of its updated parameters (the optimizer step has already zeroed the gradients).  The sample of layer
    ``i`` is the same ``DUMP_SAMPLE`` sorted positions in every run (seed ``i``), so that two builds can be compared
    value for value.  Two runs of one build do not agree bit for bit, because the token-embedding gradient is
    accumulated with floating-point atomics; on one B200 at a 1000 W power limit (GPT-2-XL, --steps 3 --warmup 2)
    the parameters differed by at most 6e-7 of the layer's largest value.  Only the first pipeline writes: after the
    all-reduce every replica holds the same layers."""
    import numpy as np
    pipeline = engine._pipeline
    if pipeline._pipeline_id != 0:
        return
    os.makedirs(directory, exist_ok=True)
    if pipeline.is_last_stage():
        np.save(os.path.join(directory, "total_loss.npy"),
                np.asarray(pipeline.execution.total_loss.detach().item(), dtype=np.float64))
    for layer in pipeline.execution._layers:
        n = layer.flat_param.numel()
        idx = np.sort(np.random.default_rng(layer.layer_id).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
        idx = torch.from_numpy(idx).to(layer.flat_param.device)
        np.save(os.path.join(directory, f"layer{layer.layer_id:03d}_param.npy"),
                layer.flat_param.detach()[idx].float().cpu().numpy())


def run_ours(args, cfg):
    import torch.distributed as dist

    from oobleck_b200 import lib as L
    from oobleck_b200.execution.dataloader import SyntheticTokenDataset
    from oobleck_b200.execution.engine import JobArguments, ModelArguments, OobleckArguments, OobleckEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"launch with torchrun --nproc-per-node {args.gpus} (WORLD_SIZE={world})"
    assert world % args.replicas == 0, "--replicas must divide --gpus"
    _quiet_nccl()
    from oobleck_b200.execution import layer as _layer
    if args.bwd_fp16 is not None:
        _layer.DEFAULT_BWD_FP16 = bool(args.bwd_fp16)
    bwd_fp16 = bool(_layer.DEFAULT_BWD_FP16) and args.nsplit == 3
    from oobleck_b200.execution import pipeline as _pipeline
    if args.fb_overlap is not None:
        _pipeline.FB_OVERLAP = bool(args.fb_overlap)
    torch.cuda.set_device(local_rank)
    L.load()
    ma = cfg["model_args"]
    T, vocab = ma["n_positions"], ma.get("vocab_size", VOCAB)
    mb, gb = cfg["microbatch"], cfg["global_batch"]
    transport_cls = None
    if world > 1:
        from oobleck_b200.execution.p2p import NvlinkRingTransport
        transport_cls = NvlinkRingTransport

    parity = None
    if args.parity_check:
        if world > 1 and not dist.is_initialized():
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        parity = parity_check(args, cfg, world, rank, local_rank, transport_cls if args.replicas == 1 else transport_cls)

    oargs = OobleckArguments(job=JobArguments(microbatch_size=mb, global_microbatch_size=gb, steps=args.steps),
                             model=ModelArguments(model_name="gpt2", model_tag=args.model, model_args=dict(ma)))
    n_samples = max(2334, gb * (args.steps + args.warmup + 2) * 2)
    dataset = SyntheticTokenDataset(num_samples=n_samples, seq_len=T, vocab_size=vocab)
    dataset.to_device(torch.device("cuda", local_rank))
    stages = world // args.replicas
    engine = OobleckEngine(local_rank, stages if args.replicas > 1 else world, 1, None, oargs, dataset=dataset,
                           nsplit=args.nsplit, transport_cls=transport_cls, device_resident=True)
    engine._world_size = world
    engine.initialize_distributed()
    engine.instantiate_pipelines(gb // mb)
    loader = engine._pipeline._dataloader
    is_last = engine._pipeline.is_last_stage()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(nsteps: int, device_resident: bool, read_loss: bool, time_gemms: bool = False):
        loader.device_resident = device_resident
        engine._pipeline.reset_iterator()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        losses = []
        e0.record()
        for i in range(nsteps):
            if time_gemms and i == nsteps - 1:
                # per-launch GEMM durations for the roofline: this one step keeps every kernel on the compute stream
                # (no wgrad side stream), so a launch's event pair times that launch alone
                L.call("oob_side_stream_enable", 0)
                fb_saved, _pipeline.FB_OVERLAP = _pipeline.FB_OVERLAP, False
                L.call("oob_gemm_timing_begin")
            engine._train_step()
            if time_gemms and i == nsteps - 1:
                L.call("oob_side_stream_enable", args.side_stream)
                _pipeline.FB_OVERLAP = fb_saved
            if read_loss and is_last:
                losses.append(float(engine._pipeline.execution.total_loss.item()))   # D2H of the step's result
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, losses

    L.call("oob_side_stream_enable", args.side_stream)
    timed(args.warmup, True, False)          # W untimed warm-up steps
    sampler = ClockSampler(local_rank)
    launches0 = L.load().oob_launch_count()
    sampler.start()
    ms, _ = timed(args.steps, True, False, time_gemms=True)
    clocks = sampler.stop()
    launches = L.load().oob_launch_count() - launches0
    g_ms, g_fl, g_ex, g_n = C.c_double(), C.c_double(), C.c_double(), C.c_long()
    L.call("oob_gemm_timing_end", C.byref(g_ms), C.byref(g_fl), C.byref(g_ex), C.byref(g_n))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, engine)
    ms_e2e, losses = timed(args.steps, False, True)

    # one more (untimed) step with CUDA events around every forward / backward pass: how busy was each stage?
    loader.device_resident = True
    engine._pipeline.reset_iterator()
    barrier()
    engine._pipeline.profile = []
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    engine._train_step()
    b1.record()
    barrier()
    step_ms = b0.elapsed_time(b1)
    busy = busy_intervals_ms(engine._pipeline.profile, b0)
    engine._pipeline.profile = None
    stage_stats = torch.tensor([busy, step_ms - busy], device="cuda")
    if world > 1:
        gathered = [torch.zeros_like(stage_stats) for _ in range(world)]
        dist.all_gather(gathered, stage_stats)
    else:
        gathered = [stage_stats]
    stage_busy = [round(float(g[0]), 2) for g in gathered]
    stage_bubble = [round(float(g[1]), 2) for g in gathered]

    last_loss = losses[-1] if losses else None
    if world > 1:   # the loss lives on the last stage(s); rank 0 prints the sum over replicas
        t = torch.tensor([last_loss if last_loss is not None else 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        last_loss = float(t.item())
    tokens_per_step = gb * T
    value = tokens_per_step * args.steps / (ms / 1e3)
    e2e = tokens_per_step * args.steps / (ms_e2e / 1e3)
    peaks = measured_peaks()
    E, Lh = ma["n_embd"], ma["num_hidden_layers"]
    fpt = flops_per_token(E, Lh, T, vocab)
    exec_tflops = (g_ex.value / (g_ms.value / 1e3) / 1e12) if g_ms.value > 0 else None
    gemm_tflops = (g_fl.value / (g_ms.value / 1e3) / 1e12) if g_ms.value > 0 else None
    template = engine._pipeline._template
    out = {
        "metric": "training_tokens_per_s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None,
        "dtype": (("f32 (fp16 x2 planes forward and backward (loss-scaled) on tcgen05, fp32 accumulate + promotion)"
                   if bwd_fp16 else
                   "f32 (fp16 x2 planes forward / bf16 x3 planes backward on tcgen05, fp32 accumulate + promotion)")
                  if args.nsplit == 3 else "split-bf16 x%d on tcgen05, fp32 accumulate" % args.nsplit),
        "data": "synthetic",
        "config": workload_config(args.model, cfg, world, args.replicas),
        "engine": {"nsplit": args.nsplit, "wgrad_side_stream": bool(args.side_stream), "bwd_fp16": bwd_fp16,
                   "fb_overlap": bool(_pipeline.FB_OVERLAP), "fb_overlap_multi_stage": bool(_pipeline.FB_OVERLAP_PP),
                   "l2": "working set per step (>6 GB of weights) far exceeds the 126 MB L2; no flush needed",
                   "stage_layers": [len(s._layer_indices) for s in template.get_stages()],
                   "stage_balance_from": engine.layer_costs_source,
                   "tensor_map_encodes": int(L.load().oob_tensor_map_encodes())},
        "parity_check": parity,
        "stage_busy_ms": stage_busy, "bubble_ms": stage_bubble,
        "clocks": clocks,
        "gpu_launches": int(launches),
        # every micro-batch crosses PCIe as the loader's three int64 [mb, T] fields (input_ids, attention_mask, labels:
        # PipelineExecution._prepare_inputs copies each dict value, pipeline.py:150-156), on the first stage of each replica
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": 3 * 8 * gb * T,
                "d2h_bytes_per_step": 4 * args.replicas, "loss": last_loss},
        "model_flops_fraction_of_bf16_peak": value * fpt / (world * peaks["bf16_tflops"] * 1e12),
        "roofline": {
            "bound": "tensor", "kernel": "gemm_bf16x3_persistent_kernel (tcgen05, all GEMM launches of the last timed step)",
            "achieved": gemm_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": (gemm_tflops / peaks["bf16_tflops"]) if gemm_tflops else None,
            "peak_source": peaks["source"] + " (cuBLAS bf16, sustained)",
            "tensor_products_per_algorithmic_flop": (g_ex.value / g_fl.value) if g_fl.value else None,
            "products_note": "GEMMs on fp16 x 2 planes issue 3 products per MAC, on bf16 x 3 planes 6: with 3 products "
                             "the algorithmic ceiling is peak / 3; executed_frac_of_peak is the tensor-pipe reading",
            "executed_tensor_tflops": exec_tflops,
            "executed_frac_of_peak": (exec_tflops / peaks["bf16_tflops"]) if exec_tflops else None,
            "launches_timed": int(g_n.value),
            "timing_note": "the last timed step runs without the wgrad side stream and without forward/backward "
                           "stream overlap, so each GEMM launch is timed alone",
            "traffic": GEMM_TRAFFIC_BYTES if args.model == "gpt2-xl" and args.nsplit == 3 and bwd_fp16 else None,
            "traffic_note": GEMM_TRAFFIC_NOTE,
        },
    }
    if world == 1 and args.cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_sample(args.model)
    if world >= RECONFIG_MIN_GPUS and args.replicas == 1 and args.with_reconfig:
        # second half of BASELINE.json's metric, AFTER the timed region: rank 0 plays the agent for a fresh set of
        # workers on the same GPUs (tools/reconfig_bench.py), SIGKILLs one inside a step and times the recovery.  The
        # other ranks wait on the host (store key, no NCCL kernel spinning on the GPUs being measured).
        torch.cuda.synchronize()
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            deadline = time.perf_counter() + EXTRAS_BUDGET_S
            try:
                out["reconfiguration"] = embedded_reconfiguration(args.model, world, deadline)
            except Exception as e:  # noqa: BLE001  (never lose the throughput line over the extra measurement)
                out["reconfiguration"] = {"error": f"{type(e).__name__}: {e}"}
            if world == 8 and CONFIG4_IN_LINE and "error" not in out["reconfiguration"].get("two_replicas", {}):
                try:
                    out["config4_dp2_x_pp4"] = embedded_config4(world, deadline)
                except Exception as e:  # noqa: BLE001
                    out["config4_dp2_x_pp4"] = {"error": f"{type(e).__name__}: {e}"}
            store.set("oob_bench_reconfig_done", "1")
        else:
            from datetime import timedelta
            try:
                store.wait(["oob_bench_reconfig_done"], timedelta(seconds=EXTRAS_BUDGET_S + 120))
            except Exception:  # noqa: BLE001
                pass
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# The driver gives one bench.py run 870 s (SCALE_r01.json per_n_timeout_s).  The extras after the timed region are bounded
# twice: each run by RECONFIG_BUDGET_S (typical: 40-60 s), all of them together by EXTRAS_BUDGET_S -- a run that would
# start with less than 45 s left is skipped and says so -- so the throughput line is printed in time whatever happens.
RECONFIG_BUDGET_S = float(os.environ.get("OOB_BENCH_RECONFIG_BUDGET_S", "150"))
EXTRAS_BUDGET_S = float(os.environ.get("OOB_BENCH_EXTRAS_BUDGET_S", "400"))
RECONFIG_MIN_GPUS = int(os.environ.get("OOB_BENCH_RECONFIG_MIN_GPUS", "4"))   # 2 replicas x >= 2 stages
TORCHRUN_ENV = ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "LOCAL_WORLD_SIZE", "GROUP_RANK",
                "GROUP_WORLD_SIZE", "ROLE_RANK", "ROLE_WORLD_SIZE", "ROLE_NAME", "OMP_NUM_THREADS",
                "TORCH_NCCL_ASYNC_ERROR_HANDLING")


CONFIG4_IN_LINE = os.environ.get("OOB_BENCH_CONFIG4", "1") == "1"


def _run_budget(deadline: float | None) -> float:
    """Seconds the next extra run may take: its own bound, cut by what is left of the extras' common budget."""
    if deadline is None:
        return RECONFIG_BUDGET_S
    return min(RECONFIG_BUDGET_S, deadline - time.perf_counter())


def _bounded_json_run(cmd: list[str], deadline: float | None) -> tuple[dict | None, dict | None, float]:
    """Run ``cmd`` in a session of its own, without anything of the surrounding torchrun in its environment, for at most
    ``_run_budget(deadline)`` seconds (the whole process group is SIGKILLed past that), and parse the last JSON line of
    its stdout.  Returns (result, problem, wall seconds): exactly one of the first two is not None; ``problem`` is
    ``{"skipped": ...}`` when the run no longer fits the budget, ``{"error": ...}`` when it overran (``"exceeded"``) or
    printed no JSON line."""
    import signal
    import subprocess
    budget = _run_budget(deadline)
    if budget < 45:
        return None, {"skipped": f"{max(budget, 0):.0f} s left of the extras' budget ({EXTRAS_BUDGET_S:.0f} s)"}, 0.0
    env = {k: v for k, v in os.environ.items() if not (k.startswith("TORCHELASTIC") or k in TORCHRUN_ENV)}
    t0 = time.perf_counter()
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, env=env, cwd=ROOT,
                         start_new_session=True, text=True)
    try:
        stdout, _ = p.communicate(timeout=budget)
    except subprocess.TimeoutExpired:
        try:
            os.killpg(p.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
        p.wait()
        return None, {"error": f"exceeded {budget:.0f} s"}, time.perf_counter() - t0
    wall = time.perf_counter() - t0
    line = next((l for l in reversed(stdout.splitlines()) if l.startswith("{")), None)
    if line is None:
        return None, {"error": f"no result (exit code {p.returncode})"}, wall
    return json.loads(line), None, wall


def embedded_config4(world: int, deadline: float | None = None) -> dict:
    """BASELINE config 4, literally: GPT-2 124M as 2 replica pipelines x 4 stages on the 8 GPUs (cross-replica gradient
    all-reduce path), measured by this very script in a torchrun of its own after the timed region of the headline run
    (``bench.py --gpus 8 --replicas 2 --model gpt2``): throughput, end-to-end throughput and the oracle parity check of
    that job.  Bounded like every extra (``_bounded_json_run``); a failure is reported, never raised."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(free_port()), os.path.join(ROOT, "bench.py"), "--gpus", str(world),
           "--replicas", "2", "--model", "gpt2", "--steps", "3", "--warmup", "3", "--cpu-baseline", "0",
           "--with-reconfig", "0"]
    r, problem, wall = _bounded_json_run(cmd, deadline)
    if problem is not None:
        return problem
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "config", "parity_check",
            "stage_busy_ms", "bubble_ms", "gpu_launches", "e2e")
    out = {k: r.get(k) for k in keep}
    out["stage_layers"] = (r.get("engine") or {}).get("stage_layers")
    out["wall_s"] = wall
    return out


def embedded_reconfiguration(model: str, world: int, deadline: float | None = None) -> dict:
    """``python tools/reconfig_bench.py`` twice in its own session: 2 replicas x world/2 stages losing a rank (BASELINE
    config 4's job; 8 GPUs: 2 x 4 -> 4 + 3) and ONE world-stage pipeline losing a rank (config 5; 8 -> 7, peer
    shadows).  Each run is bounded by RECONFIG_BUDGET_S and by what is left of the extras' common budget (``deadline``); a
    run that fails, overruns or no longer fits is reported as such."""
    out = {"metric": "reconfiguration_latency_s", "unit": "s", "higher_is_better": False,
           "definition": "lost-node message received on the worker pipe -> first completed post-reconfiguration train "
                         "step, max over the survivors (SURVEY 8d); one rank SIGKILLed inside a training step"}
    for name, replicas in (("two_replicas", 2), ("lone_pipeline", 1)):
        if replicas == 1 and world < 3:
            continue                   # a lone pipeline needs a neighbour left to restore the lost stage from
        cmd = [sys.executable, os.path.join(ROOT, "tools", "reconfig_bench.py"), "--gpus", str(world), "--replicas",
               str(replicas), "--model", model, "--steps", "5", "--kill-step", "2"]
        r, problem, wall = _bounded_json_run(cmd, deadline)
        if problem is not None:
            out[name] = problem
            if "exceeded" in problem.get("error", ""):
                break                  # do not start another run on GPUs that may still be draining
            continue
        if "error" in r:
            out[name] = {"error": str(r["error"])[:400]}
            continue
        out[name] = {"value": r["value"], "workload": r["config"]["workload"],
                     "pipelines_after": r["pipelines_after"],
                     "message_to_pipelines_rebuilt_s": r["notify_to_pipelines_rebuilt_and_states_copied_s"],
                     "replicas_identical_after": r["replicas_identical_after"],
                     "step_s_before": r["step_s_before"], "step_s_after": r["step_s_after"], "wall_s": wall}
        # training throughput of that job itself (wall clock of whole engine steps incl. the per-step votes of an
        # elastic run): with 2 replicas on 8 GPUs this is BASELINE config 4's shape (2 x 4 stages + the cross-replica
        # all-reduce) before the loss and 4 + 3 stages after it
        tps = r.get("tokens_per_step")
        for key in ("before", "after"):
            st = r.get("step_s_" + key)
            if tps and st and st.get("median"):
                out[name][f"tokens_per_s_{key}"] = tps / st["median"]
    vals = [v["value"] for v in out.values() if isinstance(v, dict) and "value" in v]
    out["value"] = max(vals) if vals else None
    return out


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant GEMM shape in the DEFAULT build (fp16 pairs
# everywhere, pair-only plane buffers): forward FC 2048 x 6400 x 1600, bias + GELU epilogue writing the fp32
# pre-activation and the two fp16 planes of GELU(x).  Source: profiles/ (see GEMM_TRAFFIC_NOTE).
GEMM_TRAFFIC_BYTES = 54.50e6 + 57.77e6
GEMM_TRAFFIC_NOTE = ("bytes/launch (dram read 54.5 MB + write 57.8 MB) from ncu --set full of the forward-FC launch in the "
                     "default pair-only build, profiles/r02_ncu_gemm_fwdfc_pair_2groups.txt; algorithmic bytes of that "
                     "launch: 54 MB of operand planes + 105 MB of outputs (part of the output is still in L2 when the "
                     "kernel ends); `achieved` aggregates all GEMM shapes")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="gpt2-xl", choices=sorted(MODELS))
    ap.add_argument("--replicas", type=int, default=1,
                    help="pipeline replicas (BASELINE config 4: --gpus 8 --replicas 2 = 2 x 4 stages + DP all-reduce)")
    ap.add_argument("--nsplit", type=int, default=3, choices=[1, 2, 3])
    ap.add_argument("--bwd-fp16", type=int, default=None, choices=[0, 1],
                    help="backward GEMMs on loss-scaled fp16 pairs (3 products) instead of bf16 x 3 (6); default: the "
                         "library default (oobleck_b200.execution.layer.DEFAULT_BWD_FP16)")
    ap.add_argument("--fb-overlap", type=int, default=None, choices=[0, 1],
                    help="forward(i+1) / backward(i) on two streams; default: oobleck_b200.execution.pipeline.FB_OVERLAP")
    ap.add_argument("--side-stream", type=int, default=1, choices=[0, 1],
                    help="0: weight-gradient kernels stay on the compute stream (A/B of the overlap)")
    ap.add_argument("--parity-check", type=int, default=1, choices=[0, 1],
                    help="check a reduced-depth model of the benchmarked width against the oracle before timing")
    ap.add_argument("--cpu-baseline", type=int, default=1, choices=[0, 1])
    ap.add_argument("--with-reconfig", type=int, default=int(os.environ.get("OOB_BENCH_RECONFIG", "1")), choices=[0, 1],
                    help="N >= 4: after the timed region, also kill a rank of a fresh job on the same GPUs and report "
                         "the recovery time under \"reconfiguration\" (adds 2-3 minutes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss and a fixed sample of every "
                         "layer's parameters) to DIR/<name>.npy")
    ap.add_argument("--reconfig", action="store_true",
                    help="reconfiguration latency after a real kill of one rank (spawns its own workers; see "
                         "tools/reconfig_bench.py)")
    args = ap.parse_args()
    cfg = MODELS[args.model]
    if args.reconfig:
        from tools.reconfig_bench import main as reconfig_main
        reconfig_main(args)
    elif args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
