#!/usr/bin/env python
"""Flagship benchmark: MNIST-DNN (simple_dnn 784-256-256-10, Adam, minibatch 300 per worker) samples/s.

    python bench.py --gpus 1 --steps 200 --warmup 20
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

One rank per GPU.  A *step* is one full parameter-server iteration of every worker: pull the master
parameters, forward + backward on a 300-row minibatch, push the gradient (ONE Adam step on the master
per push).  Weak scaling: per-GPU work is fixed, ``value`` is the whole-job samples/s.

Numbers per run (all through the public engine API, all timed on the device, max over ranks):
  value       K steps BACK TO BACK (no gap, no flush between steps: what a training loop sees) on a partition that
              lives in HBM and is larger than L2 (157 MiB): every step gathers a different 300-row minibatch by index.
              One CUDA-event pair around the K steps.
  e2e.value   the same K steps with the partition in PINNED HOST memory: every step copies its minibatch host->device
              and hands the step's loss back device->host.  One CUDA-event pair around the K steps.
  nccl_baseline_same_run / vs_baseline
              the stock PyTorch + NCCL(+cuBLAS/cuDNN) build of the same semantics (baseline/nccl_baseline.py: flat
              params, fused capturable Adam, the whole step incl. both collectives in ONE CUDA graph), measured the same
              two ways in the same process right after; ``vs_baseline`` = value / its value (BASELINE.md publishes no
              number for the reference, and the reference itself cannot run here).

``--impl reference`` would run the unmodified lifeomic/sparkflow from baseline/_ref; it needs TensorFlow
1.x + pyspark + flask + a JVM, none of which exist in this image, so it reports ``unavailable``.
``--impl nccl`` runs only the NCCL arm.

``--dump-outputs DIR`` writes what the timed `value` arm computed in its last step: every master parameter after that
step's push (``DIR/<variable name, '/' -> '.'>.npy``) and each rank's loss of that step (``DIR/loss.npy``), all float32.
Inputs and initial weights are seeded, so two builds run with the same arguments can be compared output for output.
The kernels sum bias gradients and the loss with float atomics, so two runs of one build differ by rounding, and Adam
magnifies that in parameters whose gradients are close to zero (the synthetic labels are random, so most are): three
runs of the default command on one B200 (1000 W limit) agreed in the loss to 5e-4 relative and in every parameter to
0.08 absolute.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "MNIST-DNN samples/sec (device-timed, max over ranks)"
BATCH = 300
DUMP_BYTES = 64 << 20                    # --dump-outputs budget; larger outputs are written as a fixed seeded sample
# (input dim, label dim or 0, description); the headline metric is simple_dnn, the others are BASELINE.json configs 3-5
MODELS = {
    "simple_dnn": (784, 10, "simple_dnn 784-256-256-10"),
    "cnn": (784, 10, "cnn_example conv5x5x32-pool-conv3x3x64-pool-dense10"),
    "autoencoder": (784, 0, "autoencoder_example 784-256-128-256-784"),
    "autoencoder_small": (784, 0, "autoencoder 784-32-784"),
    "wide_dnn": (4096, 1000, "wide_dnn 4096-4096x4-1000"),
}


def reference_arm(args) -> int:
    why = None
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
        import importlib

        for dep in ("tensorflow", "pyspark", "flask"):
            try:
                importlib.import_module(dep)
            except Exception as exc:
                why = f"reference needs {dep} ({type(exc).__name__}); TF-1.x/pyspark/flask/JVM are not in this image or /opt/wheelhouse"
                break
        if why is None:
            why = "reference dependencies import but the TF-1.x graph API (tf.placeholder/tf.layers/tf.Session) is required"
    except Exception as exc:  # pragma: no cover
        why = f"{type(exc).__name__}: {exc}"
    if int(os.environ.get("RANK", "0")) == 0:        # under torchrun every rank runs this: ONE line
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def _max_over_ranks(ctx, value: float) -> float:
    from sparkflow_b200.parallel import dist as D

    return max(D.all_gather_object(ctx, float(value)))


def _synthetic_partition(rows: int, seed: int, in_dim: int, n_classes: int):
    import numpy as np

    rng = np.random.default_rng(seed)
    x = rng.random((rows, in_dim), dtype=np.float32)
    y = np.eye(n_classes, dtype=np.float32)[rng.integers(0, n_classes, rows)] if n_classes else None
    return x, y


def _partition_rows(args, in_dim: int) -> int:
    rows = max(args.partition_rows, BATCH * 2)
    if in_dim * rows * 4 > (1 << 30):
        rows = max(BATCH * 2, (1 << 30) // (in_dim * 4))
    return rows


def _dump_outputs(out_dir: str, arrays: dict) -> None:
    """``arrays`` as float32 ``out_dir/<name>.npy``.  Past DUMP_BYTES in all, every array keeps the same share of its
    elements, at sorted indices drawn from a fixed seed (identical for identical shapes)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    budget = DUMP_BYTES // 4 - 1024 * len(arrays)          # elements, leaving room for the .npy headers
    total = sum(a.size for a in arrays.values())
    for name, a in arrays.items():
        if total > budget:
            keep = -(-a.size * budget // total)            # rounded up: a one-element output stays whole
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, ctx) -> dict:
    import torch

    from sparkflow_b200.models import zoo
    from sparkflow_b200.ops.optimizers import OptimizerSpec
    from sparkflow_b200.parallel import dist as D
    from sparkflow_b200.parallel.session import TrainingSession
    from sparkflow_b200.parallel.worker import B200Engine
    from sparkflow_b200.utils.clocks import ClockSampler

    dev = torch.device("cuda", ctx.local_rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    lock = args.mode == "lock"
    spec = OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.001, beta1=0.9, beta2=0.999))
    in_dim, n_classes, model_desc = MODELS[args.model]
    sess = TrainingSession(zoo.build(args.model), "x:0", "y:0" if n_classes else None, spec, acquire_lock=lock, iters=1, mini_batch=BATCH,
                           mini_stochastic_iters=1, shuffle=True, engine="b200", seed=1234, pull_mode=args.pull_mode,
                           push_mode=args.push_mode, devices=[dev.index]).open()
    eng = sess.make_engine(dev)                      # pinned-host partition: the end-to-end arm
    eng.partition_mode = "pinned"
    eng_r = B200Engine(eng.w)                        # HBM-resident partition: the back-to-back device-timed arm
    eng_r.partition_mode = "resident"
    rows = _partition_rows(args, in_dim)
    x, y = _synthetic_partition(rows, seed=100 + ctx.rank, in_dim=in_dim, n_classes=n_classes)
    eng.load_partition(x, y)
    eng_r.load_partition(x, y)
    K, W = args.steps, max(args.warmup, 3)
    n_batches = rows // BATCH
    st = eng.w.stream

    def steps(engine, n, start):
        starts = [((start + k) % n_batches) * BATCH for k in range(n)]
        engine.train_contiguous(starts, BATCH, pull=True)       # native StepDriver loop (C++), one CUDA graph per step

    def timed(engine, n, start):
        """n steps, one event pair, max over ranks; returns (ms, wall_ms)."""
        sess.sync_all()                  # drain + barrier + device-wide torch.cuda.synchronize() + barrier
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(st)
        steps(engine, n, start)
        e1.record(st)
        engine.finish()                  # stream sync + wait until the master has applied this rank's last push
        torch.cuda.synchronize(dev)
        D.barrier(ctx)
        wall = time.perf_counter() - t0
        return _max_over_ranks(ctx, e0.elapsed_time(e1)), _max_over_ranks(ctx, wall * 1e3)

    sampler = ClockSampler(dev.index or 0).start() if ctx.rank == 0 else None
    # ---------------- e2e: H2D of every minibatch + D2H of every loss ----------------
    steps(eng, W, 0)
    eng.finish()
    h2d0, d2h0 = eng.h2d_bytes, eng.d2h_bytes
    host0 = list(eng._driver.host_ns()) if getattr(eng, "_driver", None) is not None else None
    e2e_ms, wall_ms = timed(eng, K, W)
    host_us = None
    if host0 is not None:
        names = ("wait_slot", "h2d_enqueue", "event_handoff", "graph_launch", "record")
        host_us = {n: (b - a) / K / 1e3 for n, a, b in zip(names, host0, eng._driver.host_ns())}
    h2d_per_step = (eng.h2d_bytes - h2d0) // K
    d2h_per_step = (eng.d2h_bytes - d2h0) // K
    e2e_loss = eng.last_loss()

    # ---------------- value: back-to-back steps on the HBM-resident partition (> L2) ----------------
    steps(eng_r, W, 0)
    eng_r.finish()
    dev_ms, _ = timed(eng_r, K, W)
    last_loss = eng_r.last_loss()
    if args.dump_outputs:
        losses = D.all_gather_object(ctx, last_loss)
        weights = sess.weights()
        if ctx.rank == 0:
            outs = {v.name.replace("/", "."): a for v, a in zip(sess.ir.trainable, weights)}
            _dump_outputs(args.dump_outputs, dict(outs, loss=losses))
    sess.sync_all()
    # exposed push / pull per step, measured on the device (%globaltimer) inside the pull / applier kernels
    exposed = None
    if getattr(eng.w, "sharded", False):
        mine = dict(eng.w.exposed_latency(), **{"applier_" + k: v for k, v in sess.master.applier_latency().items()})
        allr = D.all_gather_object(ctx, mine)
        exposed = {k: max(r.get(k, 0) for r in allr) for k in mine}
    clocks = sampler.stop() if sampler else {}
    counters = sess.counters()
    w = eng.w
    plan_names = w.last_plan_names() if hasattr(w, "last_plan_names") else []
    launches = w.launches_per_step
    res = {
        "metric": METRIC if args.model == "simple_dnn" else f"{args.model} samples/sec (device-timed, max over ranks)",
        "value": ctx.world * BATCH * K / (dev_ms / 1e3), "unit": "samples/s", "n_gpus": ctx.world, "steps": K,
        "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "impl": "sparkflow_b200",
        "config": {"model": model_desc, "global_batch": ctx.world * BATCH, "seq_len": 1, "engine": sess.engine_kind,
                   "parallelism": f"async-ps dp{ctx.world} ({'rw-lock' if lock else 'hogwild'}, {sess.master_desc()})",
                   "optimizer": "adam(1e-3), one step per push on the master", "pull_mode": w.pull_mode, "push_mode": sess.push_mode,
                   "l2": f"no flush, steps back to back; inputs larger than L2: HBM-resident partition {rows * in_dim * 4 >> 20} MiB, every step "
                         "gathers a different minibatch (value); pinned host partition of the same size, fresh H2D every step (e2e)",
                   "kernels_per_step": plan_names, "cuda_graph": bool(w.use_graphs)},
        "e2e": {"value": ctx.world * BATCH * K / (e2e_ms / 1e3), "unit": "samples/s", "ms_per_step": e2e_ms / K,
                "h2d_bytes_per_step": int(h2d_per_step), "d2h_bytes_per_step": int(d2h_per_step), "wall_ms_per_step": wall_ms / K,
                "host_us_per_step": host_us, "final_loss": e2e_loss},
        "exposed_push_pull_us_per_step": exposed,
        "gpu_launches": int(launches * K * ctx.world),
        "clocks": clocks, "final_loss": last_loss, "master_counters": counters,
    }
    sess.close()
    return res


def run_nccl(args, ctx) -> dict:
    import torch
    import torch.distributed as dist

    from baseline.nccl_baseline import NcclBaselineWorker
    from sparkflow_b200.utils.clocks import ClockSampler

    dev = torch.device("cuda", ctx.local_rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)
    in_dim, n_classes, model_desc = MODELS[args.model]
    wk = NcclBaselineWorker(args.model, batch=BATCH, device=dev, world=ctx.world, rank=ctx.rank, use_graph=not args.baseline_eager,
                            compile=args.baseline_compile)
    rows = _partition_rows(args, in_dim)
    x, y = _synthetic_partition(rows, seed=100 + ctx.rank, in_dim=in_dim, n_classes=n_classes)
    xp = torch.from_numpy(x).pin_memory()
    yp = None if y is None else torch.from_numpy(y).pin_memory()
    xd = xp.to(dev)
    yd = None if yp is None else yp.to(dev)
    n_batches = rows // BATCH
    K, W = args.steps, max(args.warmup, 3)
    loss_host = torch.zeros(1).pin_memory()

    def step(k, host: bool):
        r = (k % n_batches) * BATCH
        wk.step((xp if host else xd)[r:r + BATCH], None if yp is None else (yp if host else yd)[r:r + BATCH])
        if host:
            loss_host.copy_(wk.loss.reshape(1), non_blocking=True)

    def timed(n, start, host):
        torch.cuda.synchronize(dev)
        if ctx.world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(n):
            step(start + k, host)
        e1.record()
        torch.cuda.synchronize(dev)
        return _max_over_ranks(ctx, e0.elapsed_time(e1))

    sampler = ClockSampler(dev.index or 0).start() if ctx.rank == 0 else None
    for k in range(W):
        step(k, True)
    e2e_ms = timed(K, W, True)
    for k in range(W):
        step(k, False)
    dev_ms = timed(K, W, False)
    clocks = sampler.stop() if sampler else {}
    torch.cuda.synchronize(dev)
    return {"metric": METRIC if args.model == "simple_dnn" else f"{args.model} samples/sec (device-timed, max over ranks)",
            "value": ctx.world * BATCH * K / (dev_ms / 1e3), "unit": "samples/s", "n_gpus": ctx.world, "steps": K,
            "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "impl": "nccl_baseline",
            "config": {"model": model_desc, "global_batch": ctx.world * BATCH, "seq_len": 1,
                       "parallelism": f"nccl broadcast/reduce dp{ctx.world}, fused Adam on rank 0", "cuda_graph": bool(wk.graphed),
                       "torch_compile": bool(wk.compiled), "capture_error": getattr(wk, "capture_error", None),
                       "l2": f"steps back to back; inputs larger than L2: device partition {rows * in_dim * 4 >> 20} MiB (value), pinned host "
                             "partition with a fresh H2D every step (e2e)"},
            "e2e": {"value": ctx.world * BATCH * K / (e2e_ms / 1e3), "unit": "samples/s", "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": BATCH * (in_dim + n_classes) * 4, "d2h_bytes_per_step": 4},
            "gpu_launches": 0, "clocks": clocks, "final_loss": float(loss_host[0])}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"])
    ap.add_argument("--model", default="simple_dnn", choices=sorted(MODELS), help="workload (the headline metric is simple_dnn)")
    ap.add_argument("--mode", default="lock", choices=["lock", "hogwild"], help="acquire_lock=True (BASELINE config 2) or Hogwild")
    ap.add_argument("--pull-mode", default=None, choices=[None, "copy", "direct"])
    ap.add_argument("--push-mode", default=None, choices=[None, "direct", "served", "sharded"],
                    help="direct: worker applies the optimizer on master memory over NVLink; served: mailbox + applier kernel "
                         "on the master GPU; sharded: master state sharded over all GPUs, one applier per shard")
    ap.add_argument("--partition-rows", type=int, default=50_100, help="rows of the per-rank partition (157 MiB > L2)")
    ap.add_argument("--no-baseline", action="store_true", help="skip the NCCL arm that normally runs in the same launch")
    ap.add_argument("--baseline-eager", action="store_true", help="NCCL arm without CUDA graphs")
    ap.add_argument("--baseline-compile", action="store_true", help="torch.compile the NCCL arm's forward/backward before capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the master parameters and the loss after the last timed step as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return reference_arm(args)
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"metric": METRIC, "error": "no CUDA device: bench.py measures the B200 engine"}))
        return 1
    from sparkflow_b200.parallel import dist as D

    ctx = D.get_context()
    if ctx.world != args.gpus:
        if ctx.rank == 0:
            print(json.dumps({"metric": METRIC, "error": f"--gpus {args.gpus} but WORLD_SIZE is {ctx.world}; launch with torchrun"}))
        return 1
    try:
        res = run_ours(args, ctx) if args.impl == "ours" else run_nccl(args, ctx)
    except Exception:
        from sparkflow_b200.ops import native

        sys.stderr.write(f"[rank {ctx.rank}] device error channel: {native.describe_device_error()}\n")
        raise
    if args.impl == "ours" and not args.no_baseline:
        try:
            base = run_nccl(args, ctx)
            res["nccl_baseline_same_run"] = {"value": base["value"], "ms_per_step": base["ms_per_step"], "e2e_value": base["e2e"]["value"],
                                             "e2e_ms_per_step": base["e2e"]["ms_per_step"],
                                             "cuda_graph": base["config"]["cuda_graph"], "torch_compile": base["config"]["torch_compile"],
                                             "final_loss": base["final_loss"]}
            res["vs_baseline"] = res["value"] / base["value"]
            res["vs_baseline_note"] = ("BASELINE.md publishes no number; ratio to the CUDA-graphed PyTorch+NCCL(+cuBLAS) build of the same "
                                       "semantics measured in this same run (nccl_baseline_same_run)")
            res["e2e"]["vs_nccl_baseline"] = res["e2e"]["value"] / base["e2e"]["value"]
        except Exception as exc:  # the headline must not die with the comparison arm
            res["nccl_baseline_same_run"] = {"error": f"{type(exc).__name__}: {exc}"}
    if ctx.rank == 0:
        print(json.dumps(res))
    D.barrier(ctx)
    return 0


if __name__ == "__main__":
    sys.exit(main())
