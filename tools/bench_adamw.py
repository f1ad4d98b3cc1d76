"""AdamW vs coupled Adam on the benchmarked step, A/B in one process; prints ONE JSON line.

    python tools/bench_adamw.py --workload resnet50x4|mlp [--steps 30 --warmup 10 --windows 4]
    torchrun --nproc-per-node N tools/bench_adamw.py --workload ...        (N > 1)

Two workers are built side by side from the same seed: ``Solver.build_worker`` with coupled Adam
(``decoupled_weight_decay=False``, what bench.py's Adam rows run) and with AdamW.  Their resident,
CUDA-graph-replayed training steps are timed in alternating windows A/B/A/B (events, warm-up,
the update kernels' own events from ``pipeline.update_events``, as bench.py does), so both see the
same clocks and neighbours.  A stock-PyTorch arm runs ``torch.optim.AdamW`` (foreach and
fused=True) under bf16 autocast, with DDP at N > 1.  At N > 1 the AdamW worker also runs
bench.py's K7-vs-NCCL parity check.  The card's name, power limit and SM clock limit come from a
read-only ``nvidia-smi --query-gpu`` in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench  # noqa: E402  (workload definitions and helpers of the headline benchmark)

LR, WD = 1e-3, 1e-5      # bench.py's Adam configuration; OptimOpts.weightDecay is the decoupled coefficient


def gpu_info(local_rank):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power, clock = [x.strip() for x in out.strip().split(",")]
        return {"name": name, "power_limit": power, "sm_clock_limit": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def build(args, ns, rank, local_rank, world, decoupled):
    import torch
    from frl_b200.solver import Solver, SolverWorkerArgs
    from frl_b200.types import Device, Precision
    t = ns.types
    torch.manual_seed(0)
    save_dir = "/tmp/frl_b200_bench_adamw_%d_%d" % (rank, int(decoupled))
    os.makedirs(save_dir, exist_ok=True)
    run_opts = t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm.ADAM, lr=LR, weightDecay=WD), batchSize=args.batch,
                         nEpochs=1, numThreads=0, singleThreaded=True, numVisualizedSamples=0)
    wargs = SolverWorkerArgs(run_opts=run_opts, problem=bench.build_problem(ns, save_dir, args), save_dir=save_dir,
                             run_device=Device.GPU, node_idx=0, node_count=1, rank=rank, local_rank=local_rank,
                             world_size=world, group_name=None, init_method="env://",
                             precision=Precision(args.precision), decoupled_weight_decay=decoupled)
    worker, _, _ = Solver.build_worker(wargs)
    worker.model.train()
    worker.criterion.train()
    return worker


def torch_arm(args, rank, local_rank, world, fused):
    """Stock torch.optim.AdamW on the same Problem and batches (bench.run_torch_gpu's step)."""
    import torch
    import torch.distributed as dist
    from frl_b200 import synthetic
    dev = torch.device("cuda", local_rank)
    ns = synthetic.api_namespace("frl_b200")
    torch.manual_seed(0)
    problem = bench.build_problem(ns, "/tmp/frl_b200_bench_adamw_torch_%d" % rank, args)
    model = problem.get_model().to(dev)
    crit = problem.get_criterion()
    mods = [m.to(dev) for m in crit.loss_modules]
    weights, names = list(crit.loss_weights), list(crit.loss_names)
    opt = torch.optim.AdamW(model.parameters(), lr=LR, weight_decay=WD, eps=1e-8, **({"fused": True} if fused else {}))
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank]) if world > 1 else model
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [bench.synthetic_batch(args, args.batch, gen, dev) for _ in range(4)]
    net.train()

    def step(data, target):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=args.precision == "bf16"):
            out = net(data)
        total = sum(w * m(o.float(), *tg) for w, m, o, tg in zip(weights, mods, out, target))
        if torch.isnan(total).any():
            raise FloatingPointError("Losses become NaN")
        opt.zero_grad()
        total.backward()
        opt.step()

    for i in range(args.warmup):
        step(*pool[i % 4])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    bench.align_ranks(world, dev)
    e0.record()
    for i in range(args.steps):
        step(*pool[i % 4])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        tv = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        ms = tv.item()
    del net, model, opt, pool
    torch.cuda.empty_cache()
    return {"optimizer": "torch.optim.AdamW(%s)" % ("fused=True" if fused else "defaults: foreach"),
            "ms_per_step": ms, "samples_per_s": world * args.batch / (ms / 1e3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="resnet50x4", choices=["mlp", "resnet50x4"])
    ap.add_argument("--steps", type=int, default=30, help="timed steps per window")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--windows", type=int, default=4, help="A/B window pairs")
    ap.add_argument("--batch", type=int, default=None, help="samples per rank per step (mlp 4096, resnet50x4 256)")
    ap.add_argument("--image", type=int, default=224)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-torch", action="store_true", help="skip the stock torch.optim.AdamW arm")
    args = ap.parse_args()
    args.batch = args.batch or bench.WORKLOADS[args.workload]["batch"]
    args.algo = "adam"
    emit = bench.claim_stdout()

    import torch
    import torch.distributed as dist
    import frl_b200  # noqa: F401
    from frl_b200 import synthetic
    from frl_b200.solver import bind_to_gpu_numa_node
    from frl_b200.solver_worker import LossLog

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    os.environ["FRL_B200_CUDA_GRAPH"] = "1"
    ns = synthetic.api_namespace("frl_b200")
    t = ns.types
    variants = {"adam": build(args, ns, rank, local_rank, world, False),
                "adamw": build(args, ns, rank, local_rank, world, True)}
    assert not variants["adam"].optimizer.decoupled and variants["adamw"].optimizer.decoupled
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [bench.synthetic_batch(args, args.batch, gen, dev) for _ in range(4)]
    W, K = args.warmup, args.steps
    n_tasks = len(variants["adam"].criterion.loss_names)
    rings = {k: LossLog(n_tasks, W + K * args.windows + 64, dev) for k in variants}
    counters = {k: 0 for k in variants}

    def step(name):
        worker, i = variants[name], counters[name]
        counters[name] += 1
        data, target = pool[i % 4]
        worker.criterion.set_step_sink(rings[name].row(i), rings[name].nan_flag)
        return worker._pass_one_minibatch(i, t.Split.TRAIN, data, target)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for name in variants:
        for _ in range(W):
            step(name)
    sync()
    ms = {k: [] for k in variants}
    for w in range(args.windows):
        for name in (("adam", "adamw") if w % 2 == 0 else ("adamw", "adam")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            bench.align_ranks(world, dev)
            e0.record()
            for _ in range(K):
                step(name)
            e1.record()
            sync()
            v = e0.elapsed_time(e1) / K
            if world > 1:
                tv = torch.tensor([v], device=dev, dtype=torch.float64)
                dist.all_reduce(tv, op=dist.ReduceOp.MAX)
                v = tv.item()
            ms[name].append(v)
    for name in variants:
        losses = rings[name].rows[:counters[name], 0]
        assert torch.isfinite(losses).all(), "non-finite loss (%s)" % name

    # the update kernels' own time: events around every update launch of 4 eager steps (in the
    # replayed graph they are nodes and carry no events), alternating between the two workers
    upd = {}
    for name, worker in variants.items():
        graphed, worker.graphed = worker.graphed, None
        worker.pipeline.update_events.clear()
        worker.pipeline.record_update_events = True
        for _ in range(6):
            step(name)
        sync()
        worker.pipeline.record_update_events = False
        worker.graphed = graphed
        ev = worker.pipeline.update_events
        per = max(len(ev) // 6, 1)
        ev = ev[2 * per:]
        launch_ms = [a.elapsed_time(b) for a, b, _, _ in ev]
        elems = sum(hi - lo for _, _, lo, hi in ev)
        bpp = bench.BYTES_PER_PARAM[("adam", args.precision)]
        upd[name] = {"update_ms_per_step": sum(launch_ms) / 4, "launches_per_step": len(ev) / 4,
                     "GBps": bpp * elems / (sum(launch_ms) / 1e3) / 1e9 if launch_ms else None,
                     "bytes_per_param": bpp}

    parity = None
    if world > 1:
        parity = bench.nvls_parity_check(variants["adamw"], lambda: step("adamw"), world, "adam", args.precision)

    def summary(v):
        s = sorted(v)
        return {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1], "windows_ms": [round(x, 4) for x in v]}

    res = {"metric": "AdamW vs coupled Adam, resident CUDA-graph-replayed step, A/B windows in one process",
           "workload": bench.workload_name(args).replace(bench.ALGO_TEXT["adam"], "Adam / AdamW lr 1e-3"),
           "world": world, "batch_per_rank": args.batch, "precision": args.precision,
           "steps_per_window": K, "warmup": W,
           "adam": dict(summary(ms["adam"]), **upd["adam"]), "adamw": dict(summary(ms["adamw"]), **upd["adamw"])}
    res["adamw_over_adam_step"] = res["adamw"]["median_ms"] / res["adam"]["median_ms"]
    if upd["adam"]["update_ms_per_step"]:
        res["adamw_over_adam_update"] = upd["adamw"]["update_ms_per_step"] / upd["adam"]["update_ms_per_step"]
    if parity is not None:
        res["parity_check"] = parity
    del variants, pool
    torch.cuda.empty_cache()
    if not args.no_torch:
        res["torch"] = [torch_arm(args, rank, local_rank, world, fused=False),
                        torch_arm(args, rank, local_rank, world, fused=True)]
        res["adamw_speedup_vs_torch_foreach"] = res["torch"][0]["ms_per_step"] / res["adamw"]["median_ms"]
    res["gpu"] = gpu_info(local_rank)
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    if world > 1:
        dist.destroy_process_group()
    if rank == 0:
        emit(json.dumps(res))


if __name__ == "__main__":
    main()
