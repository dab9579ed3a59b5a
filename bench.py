#!/usr/bin/env python
"""Flagship benchmark: GPT-2 small (double heads) data-parallel training throughput.

Metric / config are BASELINE.json's: **GPT-2 DDP tokens/sec**, bf16, synthetic PersonaChat-shaped
batches ([B, C=2, T] ids + token types + labels, [B, C] mc_token_ids, [B] mc_labels), random-init
weights, gradients all-reduced by this library's kernels, device-timed, max over ranks.
Per-GPU batch is fixed (weak scaling): B=4 (the reference's ``--train_batch_size`` default,
models/gpt2/train_gpt2_ddp.py:126), C=2 candidates, T=1024 (GPT2Config().n_positions).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference ...                     # the unmodified reference (see DESIGN.md)
    python bench.py --impl nccl ...                          # same model/engine, NCCL all-reduce
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as .npy

For N>1 launch under torchrun; with no torchrun env and N>1 the script
re-launches itself through ``python -m torch.distributed.run``.
Nothing is written into the source tree: the communicator's strategy / topology files go to a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="adapcc", choices=["adapcc", "reference", "nccl"])
    ap.add_argument("--engine", default="graph", choices=["graph", "eager", "ddp"])
    ap.add_argument("--batch", type=int, default=4, help="per-GPU batch (dialogues)")
    ap.add_argument("--candidates", type=int, default=2)
    ap.add_argument("--seq", type=int, default=1024)
    ap.add_argument("--bucket_mb", type=float, default=32.0)
    ap.add_argument("--algo", default="auto")
    ap.add_argument("--entry_point", type=int, default=-1, help="6 detect+profile, 7 profile, -1 none")
    ap.add_argument("--lm_rows", default="all", choices=["all", "scored"],
                    help="all: LM head on every position (reference behaviour, the default and the judged "
                         "number); scored: only rows whose label is not -100 (same loss and gradients)")
    ap.add_argument("--zero1", action="store_true", help="(default at N > 1; kept for old command lines)")
    ap.add_argument("--no_zero1", action="store_true",
                    help="replicated optimizer (all-reduce + full AdamW on every rank) instead of the default ZeRO-1 "
                         "sharded optimizer (reduce-scatter + AdamW on 1/N slices with the parameter broadcast fused, "
                         "multimem.st) at N > 1")
    ap.add_argument("--lm_chunk", type=int, default=0, help="rows per fused LM-head/CE chunk (0 = model default)")
    ap.add_argument("--tiny", action="store_true", help="tiny model (smoke tests only; never a bench value)")
    ap.add_argument("--ref_precision", default="bf16", choices=["bf16", "tf32", "fp32"],
                    help="--impl reference only: bf16 autocast (default, the dtype of the comparison), or the script's "
                         "literal fp32 (optionally with TF32 matmuls)")
    ap.add_argument("--relay_control", action="store_true",
                    help="--engine ddp only: negotiate the active set with the coordinator every step (straggler / relay "
                         "control, the reference's cuda_allreduce_hook behaviour); off by default in the bench")
    ap.add_argument("--allow_cpu", action="store_true", help="--impl reference only: gloo/CPU plumbing test")
    ap.add_argument("--no_nccl_arm", action="store_true",
                    help="skip the in-process NCCL arm (same engine, same buckets) that fills vs_baseline at N > 1")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0): loss.npy and "
                         "params.npy, a fixed seeded sample of the updated parameters")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs is not implemented for --impl reference")
    return a


DUMP_SAMPLE = 1 << 22          # sampled parameters: 16 MB of float32


def dump_outputs(out_dir: str, model, loss: float) -> None:
    """Writes what a caller of the training step gets back from its last call: the loss and the updated parameters
    (a sample of them), as float32 .npy files. The sample is the same for every run of a model of the same size (seeded
    indices, sorted), so two builds can be compared element for element. Compare with a tolerance: the backward pass
    accumulates some gradients with float atomics, so results differ in the last bits from run to run, and AdamW
    amplifies that over the steps."""
    import numpy as np
    import torch

    params = torch.cat([p.detach().reshape(-1).float() for p in model.parameters() if p.requires_grad])
    if params.numel() > DUMP_SAMPLE:
        g = torch.Generator().manual_seed(0)
        params = params[torch.randint(params.numel(), (DUMP_SAMPLE,), generator=g).sort().values.to(params.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))
    np.save(os.path.join(out_dir, "params.npy"), params.cpu().numpy())


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx, self.proc, self.lines, self.begin = device_index, None, [], 0

    def mark_begin(self):
        """Samples from here on count (nvidia-smi needs ~1 s to start on an 8-GPU box, so the
        process is launched long before the timed region and earlier lines are discarded)."""
        self.begin = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            import atexit

            atexit.register(self._kill)             # never leave a sampler behind if the bench dies
        except OSError:
            self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.begin:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def reference_arm(a):
    """The reference's GPT-2 arm through its own stock code path: HuggingFace ``GPT2DoubleHeadsModel(GPT2Config())``
    + torch DDP over NCCL + AdamW + clip, the step body of /root/reference/models/gpt2/train_gpt2_ddp.py:172-198
    (``baseline/reference_gpt2.py``; no repo model/kernel/engine, libadapcc.so never mapped). See DESIGN.md section 5."""
    world_env = int(os.environ.get("WORLD_SIZE", "0") or 0)
    if a.gpus > 1 and world_env == 0:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    try:
        import transformers  # noqa: F401
        from baseline import reference_gpt2
    except Exception as e:                                   # noqa: BLE001
        if int(os.environ.get("RANK", "0") or 0) == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"reference arm cannot import: {e!r}"[:300]}), flush=True)
        return 0
    return reference_gpt2.run(a, ClockSampler)


def main():
    a = parse()
    if a.impl == "reference":
        return reference_arm(a)
    world_env = int(os.environ.get("WORLD_SIZE", "0") or 0)
    if a.gpus > 1 and world_env == 0:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)

    import torch
    import torch.distributed as dist

    from adapcc_b200 import ALLREDUCE
    from adapcc_b200.adapcc import AdapCC
    from adapcc_b200.models.gpt2 import GPT2Config, GPT2DoubleHeads, synthetic_batch
    from adapcc_b200.parallel.engine import FlatDataParallel
    from adapcc_b200.runtime.native import load_library

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (CPU plumbing is covered by tests/)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    lib = load_library()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    cfg = GPT2Config.tiny() if a.tiny else GPT2Config()
    seq = min(a.seq, cfg.n_positions)
    if a.lm_chunk > 0:
        cfg.lm_chunk_rows = a.lm_chunk
    torch.manual_seed(1234)                       # same init on every rank (DDP broadcasts; we seed)
    model = GPT2DoubleHeads(cfg).to(dev)
    n_params = model.num_parameters()

    # ---- the library's public API: AdapCC.init -> setup -> communicator ---------------------------
    work = [tempfile.mkdtemp(prefix="adapcc_bench_") if rank == 0 else None]    # one directory for all ranks
    if world > 1:
        dist.broadcast_object_list(work, src=0)
    work = work[0]
    os.makedirs(os.path.join(work, "strategy"), exist_ok=True)
    grad_bytes = n_params * 2
    args = SimpleNamespace(port=5000, strategy_file=os.path.join(work, "strategy", f"bench_{world}.xml"),
                           logical_graph=os.path.join(work, "topology", f"logical_graph_{world}.xml"),
                           entry_point=a.entry_point, parallel_degree=min(4, world), profile_freq=500,
                           work_dir=work, relay_control=bool(a.relay_control and a.engine == "ddp"), algo=a.algo,
                           heap_mb=((1 if a.no_zero1 else 2) * grad_bytes >> 20) + 64, staging_mb=64, backend="nccl")
    comm = None
    comm_fn = None
    allreduce_check = None
    if a.impl == "adapcc":
        AdapCC.init(args, local, rank, world)
        AdapCC.setup(ALLREDUCE)
        comm = AdapCC.communicator.native if (world > 1 or os.environ.get("ADAPCC_FORCE_HEAP") == "1") else None
    elif world > 1:
        def comm_fn(seg):                           # NCCL baseline on the same engine / buckets
            dist.all_reduce(seg, op=dist.ReduceOp.AVG)

    tokens_per_step = a.batch * a.candidates * seq * world
    host = [synthetic_batch(a.batch, a.candidates, seq, cfg.vocab_size, seed=1000 * rank + i, pin=True)
            for i in range(4)]
    dev_batch = {k: v.to(dev) for k, v in host[0].items()}
    if a.lm_rows == "scored":
        from adapcc_b200.models.gpt2 import lm_rows_needed
        model.lm_row_capacity = max(lm_rows_needed(h["lm_labels"]) for h in host)
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    use_graph = a.engine == "graph"
    engine = None
    if a.engine == "ddp":
        # the reference's integration: torch DDP + communicator.cuda_allreduce_hook (async, side stream);
        # DDP's gradient buckets are allocated from the symmetric heap -> zero-copy all-reduce
        from adapcc_b200.parallel.ddp import rebuild_buckets, wrap_ddp

        model = model.bfloat16()
        if a.impl == "adapcc" and world > 1:
            ddp = wrap_ddp(model, AdapCC.communicator, local, bucket_cap_mb=int(a.bucket_mb))
            rebuild = lambda: rebuild_buckets(ddp, AdapCC.communicator)        # noqa: E731
        else:
            ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], bucket_cap_mb=int(a.bucket_mb),
                                                            gradient_as_bucket_view=True) if world > 1 else model
            rebuild = lambda: None                                             # noqa: E731
        opt = torch.optim.AdamW(ddp.parameters(), lr=6.25e-5, fused=True)
        it = [0]

        def ddp_step(batch):
            if a.impl == "adapcc" and world > 1:
                AdapCC.communicator.update_relay(it[0])
            loss = ddp(**batch)[0]
            opt.zero_grad(set_to_none=False)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(ddp.parameters(), 1.0)
            opt.step()
            if it[0] == 0:
                rebuild()               # DDP's one-off re-bucketing goes into the symmetric heap too
            it[0] += 1
            return loss.detach()

        step_dev = lambda: ddp_step(dev_batch)                                                   # noqa: E731
        step_e2e = lambda i: ddp_step({k: v.to(dev, non_blocking=True) for k, v in host[i % len(host)].items()})  # noqa: E731
        n_buckets, zero_copy = -1, (a.impl == "adapcc" and world > 1)
    else:
        engine = FlatDataParallel(model, comm, world_size=world, rank=rank, bucket_mb=a.bucket_mb, lr=6.25e-5,
                                  max_norm=1.0, algo=a.algo, comm_fn=comm_fn,
                                  zero1=False if a.no_zero1 else None)
        n_buckets, zero_copy = len(engine.buckets), engine.zero_copy
        if comm is not None and world > 1:
            # multi-GPU numerics of the kernel that is on the hot path, on the real bucket, against NCCL
            b0 = engine.buckets[0]
            seg = engine.flat_grad[b0.start:b0.end]
            g = torch.Generator(device=dev).manual_seed(77 + rank)
            seg.copy_(torch.randn(seg.numel(), device=dev, generator=g).to(seg.dtype))
            want = seg.float()
            dist.all_reduce(want, op=dist.ReduceOp.SUM)
            want /= world
            comm.all_reduce(seg, op="avg", algo=a.algo)
            AdapCC.communicator.synchronize()
            err = float((seg.float() - want).abs().max())
            ok = torch.tensor([1.0 if err <= 0.02 else 0.0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            allreduce_check = "ok" if float(ok.item()) == 1.0 else f"FAILED (rank {rank} max abs err {err:.4g})"
            if allreduce_check != "ok":
                raise SystemExit(f"[rank {rank}] bucket-0 all-reduce differs from NCCL: max abs err {err}")
            seg.zero_()
        if use_graph:
            engine.capture(dev_batch, warmup=2)
            step_dev = lambda: engine._graph.replay()                      # noqa: E731
            step_e2e = lambda i: engine.step_graph(host[i % len(host)])    # noqa: E731
        else:
            step_dev = lambda: engine.step(dev_batch)                      # noqa: E731
            step_e2e = lambda i: engine.step({k: v.to(dev, non_blocking=True) for k, v in host[i % len(host)].items()})  # noqa: E731

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-timed: K steps, inputs resident, CUDA events, max over ranks -------------------
    sampler.mark_begin()                          # warm-up + both timed loops run the same loaded workload
    for _ in range(max(3, a.warmup)):
        step_dev()
    barrier()
    c0 = lib.adapcc_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step_dev()
    e1.record()
    barrier()
    launches = lib.adapcc_launch_count() - c0
    if use_graph and engine is not None:
        launches = engine.native_launches_per_step * a.steps
    ms_dev = max_over_ranks(e0.elapsed_time(e1) / a.steps)

    # ---- (2) end to end: pinned-host inputs -> H2D every step, loss read back every step -----------
    for i in range(max(3, a.warmup)):
        float(step_e2e(i).item())
    barrier()
    t0 = time.perf_counter()
    e0.record()
    last = 0.0
    for i in range(a.steps):
        last = float(step_e2e(i).item())           # D2H of the step's loss (4 bytes) every step
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3) / a.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if a.dump_outputs and rank == 0:               # before the NCCL arm below re-runs the same engine
        dump_outputs(a.dump_outputs, model, last)

    zero1_flag = bool(engine is not None and getattr(engine, "zero1", False))
    if comm is not None:
        AdapCC.communicator.synchronize()
    replicas_identical = None
    if world > 1 and engine is not None:
        # data-parallel invariant after K + warm-up steps: every rank holds bit-identical parameters (a gradient that
        # missed its bucket's all-reduce would break it)
        hi, lo = engine.flat_param.float(), engine.flat_param.float()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        replicas_identical = bool(torch.equal(hi, lo))
        del hi, lo
    # ---- (3) in-process baseline arm: the SAME engine, buckets and graph over NCCL's all-reduce ----------
    ms_nccl = None
    if a.impl == "adapcc" and world > 1 and engine is not None and use_graph and not a.no_nccl_arm:
        def nccl_fn(seg):
            dist.all_reduce(seg, op=dist.ReduceOp.AVG)
        zero1_used = bool(engine.zero1)
        engine.zero1 = False                        # what stock data parallelism does: all-reduce + replicated AdamW
        engine.comm_fn = nccl_fn
        engine.capture(dev_batch, warmup=2)
        for _ in range(max(3, a.warmup)):
            engine._graph.replay()
        barrier()
        e0.record()
        for _ in range(a.steps):
            engine._graph.replay()
        e1.record()
        barrier()
        ms_nccl = max_over_ranks(e0.elapsed_time(e1) / a.steps)
    if rank == 0:
        val = tokens_per_step / (ms_dev * 1e-3)
        out = {
            "metric": "gpt2_small_ddp_train_tokens_per_sec", "value": val, "unit": "tokens/s", "n_gpus": world,
            "steps": a.steps, "warmup": max(3, a.warmup), "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": (ms_nccl / ms_dev) if ms_nccl else None, "dtype": "bf16",
            "data": "synthetic", "impl": a.impl,
            "config": {"model": "gpt2-small-double-heads (12L d768 h12 ctx1024 vocab50262, %d params)" % n_params,
                       "global_batch": a.batch * world, "per_gpu_batch": a.batch, "candidates": a.candidates,
                       "seq_len": seq, "parallelism": f"dp{world}", "engine": a.engine, "algo": a.algo,
                       "optimizer": "adamw+clip1.0 (fused)", "grad_dtype": "bf16", "zero_copy_grads": zero_copy,
                       "buckets": n_buckets, "zero1": zero1_flag,
                       "lm_rows": a.lm_rows, "lm_chunk_rows": cfg.lm_chunk_rows, "relay_control": bool(a.relay_control and a.engine == "ddp"),
                       "mlp": {0: "cublas + activation kernels", 1: "tcgen05 fused fwd", 2: "tcgen05 fused fwd+bwd"}.get(
                           getattr(model.module.h[0] if hasattr(model, "module") else model.h[0], "tc_mlp", 0), "?"),
                       "fuse_add_ln": bool(getattr(model, "fuse_add_ln", False)),
                       "l2": "working set (params+grads+optimizer state ~2 GB/step) exceeds the 126 MB L2; no flush needed"},
            "e2e": {"value": tokens_per_step / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "last_loss": last},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if allreduce_check is not None:
            out["allreduce_check"] = allreduce_check
        if replicas_identical is not None:
            out["replicas_identical"] = replicas_identical
        if ms_nccl:
            # BASELINE.md publishes no tokens/s; the practical baseline it names is "the reference-side NCCL on the
            # same box": the same engine/buckets/graph with torch.distributed's NCCL all-reduce, timed in this process
            out["baseline_arm"] = {"what": "same engine, buckets and CUDA graph over NCCL %s all-reduce (in-process)"
                                           % ".".join(map(str, torch.cuda.nccl.version())),
                                   "ms_per_step": ms_nccl, "value": tokens_per_step / (ms_nccl * 1e-3)}
        print(json.dumps(out), flush=True)
    if a.impl == "adapcc":
        AdapCC.clear(ALLREDUCE)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
