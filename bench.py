#!/usr/bin/env python
"""Headline benchmark: MNIST ConvNet DDP training throughput (images/sec, device-timed, max over
ranks) — the metric and config BASELINE.json names (ref: ddp_example.py ConvNet, batch 100/GPU,
SGD lr 1e-4, fp32 with TF32 tensor-core convolutions, synthetic MNIST-shaped data, random init).

    python bench.py --gpus N --steps K --warmup W                 # this framework
    python bench.py --impl reference --gpus N --steps K --warmup W # unmodified reference stack
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's results to DIR/*.npy

N > 1 is launched one rank per GPU by ``python -m torch.distributed.run --nproc-per-node N ...``
(RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from the environment).  Rank 0 prints ONE JSON line.

Timed regions (both arms): W >= 3 untimed warm-up steps, then exactly K steps between
barrier + torch.cuda.synchronize() on both sides, CUDA events on the launching stream, MAX over
ranks.  Inputs are seeded, so the same arguments give the same inputs on every run; ``--dump-outputs`` saves what
the last device-timed step returned (its loss) and left behind (parameters, BatchNorm buffers) for comparing two
builds output for output.  ``value`` is the device-timed step with inputs rotating through a device-resident pool that
is larger than L2 (164 MB > 126 MB).  ``e2e`` is the same step driven end to end through the framework's
own input path — ``data.MNIST`` on synthetic idx files -> ``DistributedSampler`` -> ``DataLoader(pin_memory=True)``
-> H2D of every batch -> whole-step graph -> D2H of every loss — i.e. the loop of ``cli.dist_train``
(ref: ddp_example.py:66-95).  Both arms print the same ``config`` dict; arm-specific facts live in ``details``.
The reference arm imports nothing from this package (``baseline/ref_support.py`` is standalone).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 100                    # per GPU (ref: ddp_example.py:59)
IMG = (1, 28, 28)
POOL_BATCHES = 512             # 512 x 100 x 784 x 4 B = 160.6 MB of images  > 126 MB L2
LR = 1e-4                      # ref: ddp_example.py:62
METRIC = "MNIST ConvNet DDP training throughput (images/sec, device-timed, max over ranks)"
WINDOWS = 5                    # the K timed steps are also reported as 5 back-to-back windows (min / median / max)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--syncbn", action="store_true")
    p.add_argument("--comm", default="fused", choices=["fused", "nccl"])
    p.add_argument("--no-graph", action="store_true", help="eager steps instead of the whole-step CUDA graph")
    p.add_argument("--conv-impl", default="auto", choices=["auto", "simt", "tcgen05"])
    p.add_argument("--skip-e2e", action="store_true")
    p.add_argument("--skip-verify", action="store_true", help="skip the pre-timing cross-check against torch autograd (+NCCL)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the device-timed steps, write rank 0's loss of the last step and the parameters and buffers it left "
                        "to DIR/<name>.npy (float32; integer buffers as float64)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def shared_config(world: int, syncbn: bool) -> dict:
    """The benchmark configuration — byte-identical in both arms (the driver compares it)."""
    return {"model": "ConvNet (ref ddp_example.py:22-41)", "global_batch": BATCH * world, "per_gpu_batch": BATCH, "seq_len": None,
            "parallelism": f"dp{world}", "optimizer": "SGD lr=1e-4", "syncbn": bool(syncbn),
            "inputs": f"rotating pool of {POOL_BATCHES} batches = {POOL_BATCHES * BATCH * 784 * 4 / 1e6:.0f} MB > 126 MB L2 (no explicit L2 flush)",
            "e2e_inputs": "synthetic MNIST idx files -> dataset -> DistributedSampler -> DataLoader(pin_memory) -> H2D every step"}


def window_stats(marks):
    """marks: [(steps_done, event)] recorded inside the timed region -> per-step ms of each window."""
    per = []
    for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
        if n1 > n0:
            per.append(e0.elapsed_time(e1) / (n1 - n0))
    if not per:
        return None
    return {"n": len(per), "min_ms_per_step": min(per), "median_ms_per_step": statistics.median(per), "max_ms_per_step": max(per)}


def ensure_synthetic_mnist(local_rank: int) -> str:
    """Synthetic idx files in ``<data_root>/MNIST/raw``, where both arms' MNIST datasets look for them; returns data_root.
    They live in a per-user temporary directory, not in the working directory (which may be the read-only source
    tree), and are written once and reused: their content is fixed by a seed."""
    data_root = os.path.join(tempfile.gettempdir(), f"pdt_bench_{os.getuid()}", "data")
    marker = os.path.join(data_root, "MNIST", "raw", ".synthetic_ready")
    if local_rank == 0 and not os.path.exists(marker):
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import ref_support

        ref_support.write_synthetic_mnist(data_root)
        open(marker, "w").close()
    t0 = time.time()
    while not os.path.exists(marker):
        if time.time() - t0 > 120:
            raise RuntimeError("timed out waiting for the synthetic MNIST files")
        time.sleep(0.05)
    return data_root


def snapshot_outputs(loss, module) -> dict:
    """Host copies of what a training step hands its caller: the loss it returned, and the parameters and buffers it left."""
    out = {"loss": loss}
    out.update({f"param.{k}": v for k, v in module.named_parameters()})
    out.update({f"buffer.{k}": v for k, v in module.named_buffers()})
    return {k: v.detach().cpu().clone() for k, v in out.items()}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), (t.float() if t.is_floating_point() else t.double()).numpy())


# =====================================================================================================
# this framework
# =====================================================================================================
def verify_ours(pdt, ddp, criterion, dev, rank, world, x, y):
    """Pre-timing cross-check of the whole gradient path against an independent stack: torch autograd on plain
    ``torch.nn`` modules (cuDNN / cuBLAS) holding the same weights, averaged across ranks by NCCL through
    ``torch.distributed`` (N > 1).  Also: parameters must be bit-identical on every rank.  No optimizer step is
    taken, so the timed run starts from the same weights."""
    import hashlib

    import torch
    import torch.nn as nn

    out = {"ok": False}
    module = ddp.module
    sd = {k: v.detach().clone() for k, v in module.state_dict().items()}
    oracle = nn.Module()  # same architecture as ref ddp_example.ConvNet, built from stock torch modules
    oracle.layer1 = nn.Sequential(nn.Conv2d(1, 16, 5, 1, 2), nn.BatchNorm2d(16), nn.ReLU(), nn.MaxPool2d(2, 2))
    oracle.layer2 = nn.Sequential(nn.Conv2d(16, 32, 5, 1, 2), nn.BatchNorm2d(32), nn.ReLU(), nn.MaxPool2d(2, 2))
    oracle.fc = nn.Linear(7 * 7 * 32, 10)
    oracle.to(dev)
    oracle.load_state_dict(sd)
    oracle.train()
    o = oracle.layer2(oracle.layer1(x))
    loss_ref = nn.functional.cross_entropy(oracle.fc(o.reshape(o.size(0), -1)), y)
    loss_ref.backward()
    ref_grads = torch.cat([p.grad.reshape(-1) for p in oracle.parameters()])
    if world > 1:
        import datetime

        import torch.distributed as tdist

        port = int(os.environ.get("MASTER_PORT", "29500")) + 23
        os.environ.pop("TORCHELASTIC_USE_AGENT_STORE", None)
        tdist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", world_size=world, rank=rank,
                                 timeout=datetime.timedelta(seconds=120))
        tdist.all_reduce(ref_grads)
        ref_grads /= world
        torch.cuda.synchronize()
        tdist.destroy_process_group()
    # ours: one eager forward/backward through the DDP engine (buffer broadcast + bucket allreduce included)
    bufs = {k: v.detach().clone() for k, v in module.named_buffers()}
    for p in module.parameters():
        p.grad = None
    loss = criterion(ddp(x), y)
    loss.backward()
    torch.cuda.synchronize()
    ours = torch.cat([p.grad.reshape(-1) for p in module.parameters()])
    denom = float(ref_grads.abs().max())
    out["grad_max_rel_err"] = float((ours - ref_grads).abs().max()) / max(denom, 1e-30)
    out["loss_abs_err"] = abs(float(loss.detach()) - float(loss_ref.detach()))
    with torch.no_grad():  # leave no trace: restore BN running statistics, drop the gradients
        for k, v in module.named_buffers():
            v.copy_(bufs[k])
    for p in module.parameters():
        p.grad = None
    flat = torch.cat([p.detach().reshape(-1) for p in module.parameters()]).cpu().numpy().tobytes()
    digest = hashlib.sha256(flat).hexdigest()[:16]
    digests = pdt.distributed.all_gather_object(digest) if world > 1 else [digest]
    out["param_hash"] = digest
    out["params_identical_across_ranks"] = len(set(digests)) == 1
    g2 = torch.tensor([out["grad_max_rel_err"]], device=dev)
    if world > 1:
        pdt.distributed.all_reduce(g2, pdt.distributed.ReduceOp.MAX)
    out["grad_max_rel_err"] = float(g2.item())
    out["tolerance"] = 2e-2  # TF32 convolutions on both sides, different summation orders
    out["oracle"] = "torch.nn modules + autograd (cuDNN/cuBLAS)" + (" + NCCL all_reduce / N" if world > 1 else "")
    out["ok"] = bool(out["params_identical_across_ranks"] and out["grad_max_rel_err"] < out["tolerance"] and out["loss_abs_err"] < 1e-3)
    return out


def run_ours(args):
    import torch

    import pytorch_distributed_train_b200 as pdt
    from pytorch_distributed_train_b200 import _C
    from pytorch_distributed_train_b200.engine import GraphedTrainStep
    from pytorch_distributed_train_b200.utils import ClockSampler, max_over_ranks

    rank, local_rank, world = env_rank()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if "MASTER_ADDR" not in os.environ:
        import socket

        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        init = f"tcp://127.0.0.1:{port}"
    else:
        init = "env://"
    pdt.init_process_group(backend="nccl", init_method=init, world_size=world, rank=rank, comm=args.comm)

    torch.manual_seed(0)  # identical init on every rank (ref: ddp_example.py:51)
    model = pdt.models.ConvNet()
    if args.conv_impl != "auto":
        os.environ["PDT_CONV_IMPL"] = args.conv_impl
    if args.syncbn:
        model = pdt.SyncBatchNorm.convert_sync_batchnorm(model)
    model.to(dev)
    criterion = pdt.nn.CrossEntropyLoss().to(dev)
    optimizer = pdt.optim.SGD(model.parameters(), LR)
    ddp = pdt.DistributedDataParallel(model, device_ids=[local_rank])

    # synthetic MNIST-shaped data for the device-timed number: a device-resident pool larger than L2
    g = torch.Generator().manual_seed(1234 + rank)
    dev_x = torch.rand((POOL_BATCHES, BATCH) + IMG, generator=g).to(dev)
    dev_y = torch.randint(0, 10, (POOL_BATCHES, BATCH), generator=g).to(dev)

    verify = None
    if not args.skip_verify and not args.syncbn:
        verify = verify_ours(pdt, ddp, criterion, dev, rank, world, dev_x[0], dev_y[0])

    if args.no_graph:
        def step(x, y):
            x = x.to(dev, non_blocking=True)
            y = y.to(dev, non_blocking=True)
            loss = criterion(ddp(x), y)
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            return loss
        launches_per_step = None
    else:
        graphed = GraphedTrainStep(ddp, criterion, optimizer, (dev_x[0], dev_y[0]), warmup=3, zero_grad_set_to_none=True,
                                   fuse_optimizer=os.environ.get("PDT_FUSE_OPT", "1") != "0")
        launches_per_step = graphed.kernels_per_replay
        step = graphed

    W, K = max(args.warmup, 3), args.steps

    def timed(run_step, n_warm, n_timed):
        for i in range(n_warm):
            run_step(i)
        torch.cuda.synchronize()
        pdt.distributed.barrier()
        torch.cuda.synchronize()
        marks = []
        edges = sorted({round(n_timed * w / WINDOWS) for w in range(WINDOWS + 1)})
        c0 = _C.kernel_launch_count()
        t0 = time.perf_counter()
        host_t = [0.0] * (n_timed + 1)
        for i in range(n_timed):
            if i in edges:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((i, e))
            host_t[i] = time.perf_counter()
            run_step(n_warm + i)
        host_t[n_timed] = time.perf_counter()
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        marks.append((n_timed, e))
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        pdt.distributed.barrier()
        torch.cuda.synchronize()
        ws = window_stats(marks)
        if ws is not None:  # host-side view: the slowest individual steps (index, ms) — loader stalls / GIL hand-offs show up here
            per = sorted(((host_t[i + 1] - host_t[i]) * 1e3, i) for i in range(n_timed))
            ws["host_median_ms_per_step"] = per[len(per) // 2][0]
            ws["host_slowest_steps"] = [(i, round(ms, 3)) for ms, i in per[-3:]]
        return marks[0][1].elapsed_time(marks[-1][1]), wall_ms, _C.kernel_launch_count() - c0, ws

    # ---- device-timed steps, inputs rotate through a device pool larger than L2 ------------------------
    last = {}

    resident = {} if args.no_graph else {"inputs_ready": True}   # the pool is a GPU-resident dataset: complete long before the step

    def dev_step(i):
        j = i % POOL_BATCHES
        last["loss"] = step(dev_x[j], dev_y[j], **resident)

    with ClockSampler(gpu_index=local_rank, period_ms=100) as clocks:
        ms_dev, _, eager_launches, windows = timed(dev_step, W, K)
        final_loss = float(last["loss"].detach())
        # taken before the e2e run below trains the same model further (and replays overwrite the graph's loss tensor)
        outputs = snapshot_outputs(last["loss"], ddp.module) if args.dump_outputs and rank == 0 else None
        # ---- end to end through the framework's own input path (the loop of cli.dist_train) -----------
        e2e = None
        if not args.skip_e2e:
            data_root = ensure_synthetic_mnist(local_rank)
            dataset = pdt.data.MNIST(root=data_root, train=True)
            sampler = pdt.DistributedSampler(dataset, num_replicas=world, rank=rank)
            loader = pdt.DataLoader(dataset=dataset, batch_size=BATCH, shuffle=False, num_workers=0, pin_memory=True, sampler=sampler,
                                    prefetch=int(os.environ.get("PDT_BENCH_PREFETCH", "8")))
            R = 8
            host_loss = torch.zeros(R, dtype=torch.float32).pin_memory()
            evs = [torch.cuda.Event() for _ in range(R)]
            state = {"h2d": 0, "logged": 0.0}

            def batches():
                while True:  # epochs, like the reference's outer loop (ref: ddp_example.py:81)
                    for b in loader:
                        if b[0].shape[0] == BATCH:
                            yield b

            it = batches()

            stall = {"loader": (0.0, -1), "step": (0.0, -1), "readback": (0.0, -1)}
            host_samples = {"loader": [], "step": [], "readback": []}

            pending = {"log": None}

            def e2e_step(i):
                t0 = time.perf_counter()
                images, labels = next(it)                     # pinned host tensors from the loader
                t1 = time.perf_counter()
                state["h2d"] = images.numel() * images.element_size() + labels.numel() * labels.element_size()
                loss = step(images, labels)                   # H2D of this batch into the step's inputs + graph replay
                t2 = time.perf_counter()
                if args.no_graph:
                    if i >= R:
                        evs[i % R].synchronize()                  # the slot's previous loss has reached the host
                    host_loss[i % R].copy_(loss.detach(), non_blocking=True)   # D2H of every step's loss
                    evs[i % R].record()
                    if (i + 1) % 10 == 0 and rank == 0:           # the reference's logging cadence: a blocking read (ref: ddp_example.py:93-95)
                        evs[i % R].synchronize()
                        state["logged"] = float(host_loss[i % R])
                else:
                    h = step.loss_to_host()                       # D2H of every step's loss (side stream, pinned ring)
                    if pending["log"] is not None:                # the log line of step i-1 (ref cadence: every 10th step, ddp_example.py:93-95):
                        state["logged"] = pending["log"].item()   # blocking read, issued after step i is queued so the device stays busy
                        pending["log"] = None
                    if (i + 1) % 10 == 0 and rank == 0:
                        pending["log"] = h
                    state["last"] = h
                t3 = time.perf_counter()
                if i >= W:   # where the host spends its time: worst moments (ms, timed step index) and per-phase samples for the medians
                    for k, d in (("loader", t1 - t0), ("step", t2 - t1), ("readback", t3 - t2)):
                        host_samples[k].append(d * 1e3)
                        if d * 1e3 > stall[k][0]:
                            stall[k] = (round(d * 1e3, 3), i - W)

            ms_e2e_dev, ms_e2e_wall, _, e2e_windows = timed(e2e_step, W, K)
            if e2e_windows is not None:
                e2e_windows["host_worst_ms"] = stall
                e2e_windows["host_median_ms"] = {k: round(sorted(v)[len(v) // 2], 4) for k, v in host_samples.items() if v}
                e2e_windows["host_cpus"] = len(os.sched_getaffinity(0))
            e2e = {"ms": max(ms_e2e_dev, ms_e2e_wall), "dev_ms": ms_e2e_dev, "wall_ms": ms_e2e_wall, "windows": e2e_windows,
                   "h2d": state["h2d"], "loss": float(host_loss[(W + K - 1) % R]) if args.no_graph else state["last"].item()}
    ms_dev = max_over_ranks(ms_dev)
    out = None
    if e2e is not None:
        e2e["ms"] = max_over_ranks(e2e["ms"])
    if rank == 0:
        imgs = BATCH * world * K
        value = imgs / (ms_dev / 1e3)
        info = ddp._get_ddp_logging_data()
        gpu_launches = (launches_per_step * K) if launches_per_step is not None else eager_launches
        out = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32 (tf32 tensor-core conv, fp32 accumulate) — the reference's precision",
            "data": "synthetic MNIST-shaped images, random-init weights",
            "impl": "ours",
            "config": shared_config(world, args.syncbn),
            "details": {"comm": info.get("comm_kind"), "cuda_graph": not args.no_graph, "buckets": info.get("bucket_sizes"),
                        "grad_copies_into_bucket": info.get("copies_into_bucket"),
                        "fused_allreduce_sgd": bool(getattr(optimizer, "_fused_active", False)),
                        "optimizer_step": ("inside the gradient-reduce kernels (allreduce + SGD per chunk; tests/test_gpu_multigpu.py::test_fused_allreduce_sgd)"
                                           if getattr(optimizer, "_fused_active", False) else
                                           "inside the last backward kernel (SgdRider; tests/test_gpu_kernels.py::test_optimizer_rides_on_the_last_backward_kernel)"
                                           if (not args.no_graph and launches_per_step == 3) else "separate multi-tensor SGD kernel"),
                        "reduce_chunks": info.get("reduce_chunks"), "backward_comm_exposed_us": (info.get("avg_backward_comm_exposed_time_us") if info.get("timed_iterations") else None),  # eager iterations past the reducer's 10-step warm-up only; a replayed graph carries no marks
                        "input_staging": ("double-buffered: the copy of batch k+1 into the step's input buffers (D2D from the resident pool / H2D "
                                          "from pinned memory in e2e) runs on a copy stream while step k replays; every step still copies its "
                                          "own batch" if (not args.no_graph and getattr(graphed, "double_buffer", False)) else "copied on the compute stream in front of the step")},
            "windows": windows,
            "gpu_launches": int(gpu_launches),
            "gpu_launches_per_step": launches_per_step if launches_per_step is not None else eager_launches / K,
            "clocks": {k: v for k, v in clocks.summary().items() if k in ("sm_mhz", "sm_max_mhz", "reasons", "power_w_max", "samples")},
            "final_loss": final_loss,
        }
        if verify is not None:
            out["verify"] = verify
        if e2e is not None:
            out["e2e"] = {"value": imgs / (e2e["ms"] / 1e3), "unit": "images/s", "ms_per_step": e2e["ms"] / K,
                          "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": 4, "windows": e2e["windows"],
                          "device_ms_per_step": e2e["dev_ms"] / K, "wall_ms_per_step": e2e["wall_ms"] / K,
                          "note": "pdt.data.MNIST(synthetic idx files) -> pdt.DistributedSampler -> pdt.DataLoader(batch 100, pin_memory) -> "
                                  "GraphedTrainStep(pinned images, pinned labels): H2D + whole-step graph replay; step.loss_to_host(): async D2H of every "
                                  "loss; blocking read of every 10th loss on rank 0, issued after the following step has been queued (the loop of "
                                  "cli.dist_train; cadence of ref ddp_example.py:93-95)"}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    pdt.destroy_process_group()
    if verify is not None and not verify["ok"]:
        if out is not None:
            print(json.dumps(out), flush=True)
        raise SystemExit(f"[rank {rank}] verification against torch autograd/NCCL failed: {verify}")
    return out


# =====================================================================================================
# reference arm: the unmodified reference from baseline/_ref, its own code path, nothing of ours imported
# =====================================================================================================
def _ensure_reference():
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    if not os.path.exists(os.path.join(ref_dir, "ddp_example.py")):   # installed by build(); the benchmark does not write the tree
        raise FileNotFoundError(f"{ref_dir} has no ddp_example.py; build() installs the reference there")
    return ref_dir


def run_reference(args):
    try:
        ref_dir = _ensure_reference()
        sys.path.insert(0, ref_dir)
        import ddp_example as ref  # noqa: F401  (unmodified copy of /root/reference/ddp_example.py)
        import ref_support         # standalone harness helpers (no import of our package)
    except Exception as e:  # noqa: BLE001
        return {"impl": "reference", "unavailable": f"reference not importable: {type(e).__name__}: {e}"[:300]}
    import torch
    import torch.distributed as dist
    import torch.nn as nn

    rank, local_rank, world = env_rank()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    import faulthandler

    faulthandler.dump_traceback_later(240, repeat=True, file=sys.stderr)  # say where we are if something wedges
    W, K = max(args.warmup, 3), args.steps
    base_port = int(os.environ.get("MASTER_PORT", "29500"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(local_rank)

    # The reference rendezvouses over its own tcp:// endpoint (ddp_example.py:55); under torchrun the
    # TORCHELASTIC_USE_AGENT_STORE flag would make *every* rank a client of that port (nobody serves it).
    os.environ.pop("TORCHELASTIC_USE_AGENT_STORE", None)
    # ---- (1) stack-only: the reference's model / DDP / loss / optimizer with device-resident inputs ----
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{base_port + 11}", world_size=world, rank=rank)
    torch.manual_seed(0)
    model = ref.ConvNet()
    if args.syncbn:
        model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
    model.cuda(local_rank)
    criterion = nn.CrossEntropyLoss().cuda(local_rank)
    optimizer = torch.optim.SGD(model.parameters(), LR)
    model = nn.parallel.DistributedDataParallel(model, device_ids=[local_rank])
    g = torch.Generator().manual_seed(1234 + rank)
    dev_x = torch.rand((POOL_BATCHES, BATCH) + IMG, generator=g).to(dev)
    dev_y = torch.randint(0, 10, (POOL_BATCHES, BATCH), generator=g).to(dev)

    def ref_step(i):
        j = i % POOL_BATCHES
        outputs = model(dev_x[j])
        loss = criterion(outputs, dev_y[j])
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        return loss

    with ref_support.Clocks(gpu_index=local_rank) as clocks:
        for i in range(W):
            ref_step(i)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        marks = []
        edges = sorted({round(K * w / WINDOWS) for w in range(WINDOWS + 1)})
        for i in range(K):
            if i in edges:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((i, e))
            loss = ref_step(W + i)
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        marks.append((K, e))
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([marks[0][1].elapsed_time(marks[-1][1])], device=dev)
        dist.all_reduce(t, dist.ReduceOp.MAX)
        ms_dev = float(t.item())
        windows = window_stats(marks)
        final_loss = float(loss.detach())
        outputs = snapshot_outputs(loss, model.module) if args.dump_outputs and rank == 0 else None
        del model, optimizer
        dist.destroy_process_group()

        # ---- (2) end to end: ddp_example.dist_train itself, untouched ---------------------------------
        # Offline substitutes for what the script fetches/assumes: synthetic idx files where torchvision's
        # MNIST expects them (./data/MNIST/raw), loopback init address.  Timing is injected by wrapping the
        # DataLoader iterator (a torch class, not reference code): sync + barrier + event at step W and W+K.
        e2e_ms = None
        e2e_err = None
        if not args.skip_e2e:
            try:
                data_root = ensure_synthetic_mnist(local_rank)
                e2e_ms = _reference_e2e(ref, args, rank, local_rank, world, W, K, base_port + 12, data_root)
            except Exception as e:  # noqa: BLE001
                e2e_err = f"{type(e).__name__}: {e}"[:300]
    if rank != 0:
        return None
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    imgs = BATCH * world * K
    out = {
        "metric": METRIC, "value": imgs / (ms_dev / 1e3), "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32 (torch defaults: TF32 allowed in cuDNN conv, fp32 matmul)", "data": "synthetic MNIST-shaped images, random-init weights",
        "impl": "reference",
        "config": shared_config(world, args.syncbn),
        "details": {"stack": f"torch {torch.__version__} DistributedDataParallel + NCCL {'.'.join(map(str, torch.cuda.nccl.version()))} + cuDNN/cuBLAS",
                    "model_class": "ddp_example.ConvNet (baseline/_ref, unmodified)"},
        "windows": windows,
        "gpu_launches": 0, "clocks": clocks.summary(), "final_loss": final_loss,
    }
    if e2e_ms is not None:
        out["e2e"] = {"value": imgs / (e2e_ms / 1e3), "unit": "images/s", "ms_per_step": e2e_ms / K,
                      "h2d_bytes_per_step": BATCH * 784 * 4 + BATCH * 8, "d2h_bytes_per_step": 0.4,
                      "note": "ddp_example.dist_train() unmodified: torchvision MNIST (PIL per sample) + DistributedSampler + DataLoader(pin_memory) + .cuda(non_blocking) + loss.item() every 10 steps"}
    elif e2e_err:
        out["e2e_error"] = e2e_err
    return out


def _reference_e2e(ref, args, rank, local_rank, world, W, K, port, data_root):
    import io
    from contextlib import redirect_stdout
    from types import SimpleNamespace

    import torch
    import torch.distributed as dist
    import torch.utils.data as tud

    steps_per_epoch = -(-(-(-60000 // world)) // BATCH)  # ceil(ceil(60000/world)/100): 600/300/150/75
    epochs = -(-(W + K + 1) // steps_per_epoch)
    state = {"n": 0, "start": None, "end": None, "ms": None}
    Base = tud.DataLoader

    class TimedLoader(Base):
        def __iter__(self):
            for batch in super().__iter__():
                if state["n"] == W:
                    torch.cuda.synchronize()
                    dist.barrier()
                    torch.cuda.synchronize()
                    state["start"] = torch.cuda.Event(enable_timing=True)
                    state["start"].record()
                if state["n"] == W + K:
                    state["end"] = torch.cuda.Event(enable_timing=True)
                    state["end"].record()
                    torch.cuda.synchronize()
                    dist.barrier()
                    state["ms"] = state["start"].elapsed_time(state["end"])
                    return  # enough: let the epoch (and dist_train) finish
                if state["ms"] is not None:
                    return
                state["n"] += 1
                yield batch

    ns = SimpleNamespace(gpus=world, epochs=epochs, backend="nccl", syncbn=args.syncbn, world_size=world,
                         init_method=f"tcp://127.0.0.1:{port}")
    tud.DataLoader = TimedLoader
    cwd = os.getcwd()
    os.chdir(os.path.dirname(data_root))   # the reference reads MNIST from ./data
    try:
        buf = io.StringIO()
        with redirect_stdout(buf):   # the reference prints every 10 steps; keep our stdout to one JSON line
            ref.dist_train(local_rank, ns)
    finally:
        os.chdir(cwd)
        tud.DataLoader = Base
    if state["ms"] is None:
        raise RuntimeError(f"reference loop ended after {state['n']} steps, before warmup+steps={W + K}")
    t = torch.tensor([state["ms"]], device=torch.device("cuda", local_rank))
    dist.all_reduce(t, dist.ReduceOp.MAX)
    ms = float(t.item())
    dist.destroy_process_group()
    return ms


def main():
    args = parse()
    if args.impl == "reference":
        out = run_reference(args)
    else:
        out = run_ours(args)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
