#!/usr/bin/env python
"""Headline benchmark: samples/sec of the data-parallel training step on the synthetic 2-task
MLP Problem (BASELINE.json configs[1] at N=1, configs[2] at N>1; batch 4096 per rank).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 path
    python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on host CPU
    python bench.py --impl torch-gpu --gpus N ...            # stock PyTorch on the GPU: autocast +
                                                             # torch.optim (+ DDP at N>1), the
                                                             # "kernel to beat" of SURVEY §8(d)
    python bench.py --workload resnet18|resnet50x4 ...       # BASELINE configs[3] / configs[4]
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's
                                                             # outputs as DIR/*.npy (float32)

One JSON line on stdout (rank 0).  Everything else goes to stderr.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "samples/sec (whole box) on synthetic 2-task Problem"
WIDTH, N_CLASSES, REG_DIM, DEPTH = 4096, 1000, 64, 3


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch-gpu"])
    ap.add_argument("--workload", default="mlp", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", default=None, choices=["sgd", "adam", "rmsprop"],
                    help="default: the workload's (mlp/resnet18 sgd, resnet50x4 adam)")
    ap.add_argument("--batch", type=int, default=None, help="samples per rank per step (mlp 4096, resnets 256)")
    ap.add_argument("--image", type=int, default=224, help="resnet workloads: image side")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-batch", type=int, default=None,
                    help="CPU arm: samples per step (default: the workload's batch for --impl reference, "
                         "a bounded sample — mlp 1024, resnets 32 — for the in-line cpu_baseline leg)")
    ap.add_argument("--torch-optim", default="default", choices=["default", "fused"],
                    help="torch-gpu arm: torch.optim as the reference builds it (foreach) or fused=True")
    ap.add_argument("--no-torch-baseline", action="store_true",
                    help="b200 arm: skip the in-process stock-PyTorch-GPU comparison")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="b200 arm, N>1: skip the K7-vs-NCCL self-check after the timed region")
    ap.add_argument("--cpu-steps", type=int, default=3, help="cpu_baseline leg: timed steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--bucket-mb", type=float, default=None, help="gradient bucket cap (MiB)")
    ap.add_argument("--graph", type=int, default=1, help="replay the step from a CUDA graph (1) or issue it eagerly (0)")
    ap.add_argument("--profile", default=None,
                    help="write a JSON summary (device time per kernel per step, torch.profiler over 5 steps) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="b200 arm: after the timed steps, write what the last timed step returned (model "
                         "outputs, losses) and a fixed sample of the master weights it left as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs is implemented for --impl b200 only")
    wl = WORKLOADS[args.workload]
    if args.algo is None:
        args.algo = wl["algo"]
    if args.batch is None:
        args.batch = wl["batch"]
    return args


# --------------------------------------------------------------------------------------------------
# shared: the Problem
# --------------------------------------------------------------------------------------------------

WORKLOADS = {
    # BASELINE.json configs[1]/[2] (the metric's configuration), configs[3], configs[4]
    "mlp": {"algo": "sgd", "batch": 4096, "cpu_sample_batch": 1024, "params": 54_703_144,
            "what": "2-task MLP Problem: 4096-d in, 3x[Linear(4096,4096)+ReLU] trunk, heads 4096->1000 CE + "
                    "4096->64 MSE (54.70M params)"},
    "resnet18": {"algo": "sgd", "batch": 256, "cpu_sample_batch": 32, "params": 11_689_512,
                 "what": "single-task ResNet-18 Problem: torchvision resnet18 trunk + Linear(512,1000) CE head "
                         "(11.69M params, 62 tensors), synthetic 3x%dx%d images"},
    "resnet50x4": {"algo": "adam", "batch": 256, "cpu_sample_batch": 16, "params": 25_790_618,
                   "what": "4-task Problem over a shared ResNet-50 trunk: heads 2048->{1000 CE, 100 CE, 10 MSE, "
                           "4 MSE} (25.79M params, 167 tensors), synthetic 3x%dx%d images"},
}
ALGO_TEXT = {"sgd": "SGD momentum 0.9 lr 0.01", "adam": "Adam lr 1e-3 (L2-coupled, as the reference)",
             "rmsprop": "RMSprop momentum 0.9 lr 1e-3"}


def workload_name(args, batch=None):
    what = WORKLOADS[args.workload]["what"]
    if "%d" in what:
        what = what % (args.image, args.image)
    return "%s, batch %d/rank, %s wd=1e-5" % (what, batch or args.batch, ALGO_TEXT[args.algo])


def build_problem(ns, save_dir, args, n_train=64, pinned=False, fast_fields=False, uint8=False):
    from frl_b200 import synthetic
    if args.workload == "mlp":
        return synthetic.make_mlp_problem(ns, save_dir, n_train=n_train, width=WIDTH, n_classes=N_CLASSES,
                                          reg_dim=REG_DIM, depth=DEPTH, pinned=pinned, fast_fields=fast_fields)
    return synthetic.make_resnet_problem(ns, save_dir, args.workload, image=args.image, n_train=n_train,
                                         pinned=pinned, uint8=uint8)


def synthetic_batch(args, batch, gen, device):
    """One (data, target) minibatch of the workload's shape, generated on ``device``."""
    import torch
    from frl_b200 import synthetic
    if args.workload == "mlp":
        x = torch.randn(batch, WIDTH, device=device, generator=gen)
        y = torch.randint(0, N_CLASSES, (batch,), device=device, generator=gen)
        r = torch.randn(batch, REG_DIM, device=device, generator=gen)
        return [x], [(y,), (r,)]
    x = torch.randn(batch, 3, args.image, args.image, device=device, generator=gen)
    target = []
    for kind, dim, _, _ in synthetic.RESNET_CONFIGS[args.workload][1]:
        if kind == "cls":
            target.append((torch.randint(0, dim, (batch,), device=device, generator=gen),))
        else:
            target.append((torch.randn(batch, dim, device=device, generator=gen),))
    return [x], target


def run_opts_for(ns, algo, batch):
    t = ns.types
    lr = 0.01 if algo == "sgd" else 1e-3
    return t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm(algo), lr=lr), batchSize=batch,
                     nEpochs=1, numThreads=0, singleThreaded=True, numVisualizedSamples=0)


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/_ref) or its restatement (oracle/ref_loop) on the host cores
# --------------------------------------------------------------------------------------------------

def time_cpu_reference(args, batch, steps, warmup):
    """The reference's `_pass_one_minibatch` on the host cores, on a bounded sample of the workload.

    kind "reference": the UNMODIFIED reference (packed by oracle/build_ref.py into oracle/_ref,
    imported as frldistml.scaffold) — its own SolverWorker, criteria and `_create_optimizer` on
    the synthetic Problem instantiated against ITS plugin API, `cpuonly`;
    kind "port": oracle/ref_loop.reference_minibatch (the restatement) when oracle/_ref is absent."""
    import torch
    import frl_b200  # noqa: F401  (only the synthetic Problem definition)
    from frl_b200 import synthetic
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 by default)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except AttributeError:
        torch.set_num_threads(os.cpu_count() or 1)
    from oracle import ref_shim
    g = torch.Generator().manual_seed(1234)
    data, target = synthetic_batch(args, batch, g, torch.device("cpu"))
    lr = 0.01 if args.algo == "sgd" else 1e-3
    if ref_shim.reference_available():
        ref_shim.import_reference()
        ns = synthetic.api_namespace("frldistml.scaffold")
        from frldistml.scaffold import solver as ref_solver
        from frldistml.scaffold import solver_worker as ref_sw
        t = ns.types
        torch.manual_seed(0)
        problem = build_problem(ns, "/tmp/frl_b200_bench_cpu", args)
        model, crit = problem.get_model(), problem.get_criterion()
        run_opts = t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm(args.algo), lr=lr), batchSize=batch,
                             nEpochs=1, numThreads=0, singleThreaded=True, cpuonly=True,
                             numVisualizedSamples=0)
        from itertools import chain
        opt = ref_solver._create_optimizer(chain(model.parameters(), crit.parameters()), run_opts.optim)
        # the dataset cache is an out-of-scope subsystem the minibatch never touches: hand the
        # constructor the one attribute it checks instead of 85 % of the host's RAM
        from types import SimpleNamespace
        worker = ref_sw.SolverWorker(model, crit, opt, torch.device("cpu"), run_opts,
                                     SimpleNamespace(local_worker_count=1),
                                     local_rank=0, node_idx=0, node_count=1)
        model.train()
        crit.train()

        def step(i):
            worker._pass_one_minibatch(i, t.Split.TRAIN, data, target)

        kind = "reference"
        how = ("the unmodified reference's SolverWorker._pass_one_minibatch (oracle/_ref, torch %s CPU ops + "
               "torch.optim)" % torch.__version__)
    else:
        from oracle import ref_loop
        ns = synthetic.api_namespace("frl_b200")
        torch.manual_seed(0)
        problem = build_problem(ns, "/tmp/frl_b200_bench_cpu", args)
        model, crit = problem.get_model(), problem.get_criterion()
        mods, weights, names = list(crit.loss_modules), list(crit.loss_weights), list(crit.loss_names)
        params = list(model.parameters())
        opt = ref_loop.make_optimizer(params, ref_loop.OptimSpec(algo=args.algo, lr=lr))
        model.train()

        def step(i):
            ref_loop.reference_minibatch(
                model, lambda o, tg: ref_loop.parallel_criterion(mods, weights, names, o, tg), opt, params,
                0.0, data, target)

        kind = "port"
        how = "oracle/ref_loop.reference_minibatch (stock torch CPU ops + torch.optim)"
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step(i)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": batch * steps / total, "unit": "samples/s", "cores": torch.get_num_threads(),
            "host_cpus": os.cpu_count(), "kind": kind, "batch": batch,
            "sample": "%d timed steps (+%d warm-up) of the same workload at batch %d, fp32, %s" % (
                steps, warmup, batch, how),
            "ms_per_step": 1e3 * total / steps, "step_p50_ms": 1e3 * statistics.median(times)}


def main_reference(args, rank):
    if rank != 0:
        return
    # the driver's reference arm runs the metric's own configuration (same batch as the b200 arm)
    # unless a smaller bounded sample is asked for
    batch = args.cpu_batch or args.batch
    res = time_cpu_reference(args, batch, args.steps, args.warmup)
    note = "reference implementation on the host CPU, fp32"
    if batch != args.batch:
        note += "; bounded sample: batch %d per step instead of %d" % (batch, args.batch)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "step_p50_ms": res["step_p50_ms"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            # the b200 arm's workload keys (the job this CPU sample stands for) + what was run
            "config": {"workload": workload_name(args, batch), "global_batch": args.batch * args.gpus,
                       "parallelism": "dp%d" % args.gpus, "note": note},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------

class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                      # noqa: BLE001
            log("clock sampling unavailable:", e)
            self._nv = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:                       # noqa: BLE001
                pass
            self._stop.wait(0.004)

    def __enter__(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------
# stock-PyTorch-GPU arm: what the reference does on a GPU (SURVEY §8d "kernel to beat")
# --------------------------------------------------------------------------------------------------

def run_torch_gpu(args, rank, local_rank, world, steps, warmup, with_e2e=True, profile_path=None):
    """The reference's GPU training step with stock PyTorch only (reference solver.py:162-188
    `_create_optimizer` = torch.optim defaults, :265-294 DistributedDataParallel(device_ids=[rank])
    at world > 1; solver_worker.py:551-592 forward / criterion / isnan / zero_grad / backward /
    step) on the same Problem, batch and synthetic data as the b200 arm.  `--precision bf16` runs
    the forward under torch.autocast(bfloat16) with fp32 parameters and optimizer state — the same
    numerical recipe as this repo's BF16 mode; fp32 is the reference's literal configuration.
    Nothing of this repo's kernels, arena or pipeline is on this path (only the synthetic Problem
    definition, instantiated on the package's plugin API)."""
    import torch
    import torch.distributed as dist
    import frl_b200  # noqa: F401
    from frl_b200 import synthetic

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ns = synthetic.api_namespace("frl_b200")
    B = args.batch
    torch.manual_seed(0)
    problem = build_problem(ns, "/tmp/frl_b200_bench_torch_%d" % rank, args)
    model = problem.get_model().to(dev)
    crit = problem.get_criterion()
    mods = [m.to(dev) for m in crit.loss_modules]
    weights, names = list(crit.loss_weights), list(crit.loss_names)
    lr = 0.01 if args.algo == "sgd" else 1e-3
    kw = {"fused": True} if args.torch_optim == "fused" else {}
    params = list(model.parameters())
    if args.algo == "sgd":
        opt = torch.optim.SGD(params, lr=lr, momentum=0.9, weight_decay=1e-5, **kw)
    elif args.algo == "adam":
        opt = torch.optim.Adam(params, lr=lr, weight_decay=1e-5, eps=1e-8, **kw)
    else:
        opt = torch.optim.RMSprop(params, lr=lr, momentum=0.9, weight_decay=1e-5)
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank])
    autocast = args.precision == "bf16"
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [synthetic_batch(args, B, gen, dev) for _ in range(4)]
    net.train()

    def step(data, target):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            out = net(data)
        split = {n: w * m(o.float(), *t) for n, w, m, o, t in zip(names, weights, mods, out, target)}
        total = sum(split.values())
        if torch.isnan(total).any():                 # the reference's per-step host sync (:569)
            raise FloatingPointError("Losses become NaN")
        opt.zero_grad()
        total.backward()
        opt.step()
        return total

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        tv = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        return tv.item()

    for i in range(warmup):
        step(*pool[i % 4])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    align_ranks(world, dev)
    e0.record()
    for i in range(steps):
        step(*pool[i % 4])
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    res = {"value": world * B / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms,
           "optimizer": "torch.optim.%s(%s)" % (type(opt).__name__, "fused=True" if kw else "defaults: foreach"),
           "grad_sync": "DistributedDataParallel + NCCL" if world > 1 else "none (1 GPU)",
           "precision": "torch.autocast(bfloat16) forward, fp32 parameters/gradients/state" if autocast else "fp32",
           "step": "eager launches incl. the reference's isnan host sync"}
    if profile_path and rank == 0 or (profile_path and world > 1):
        from contextlib import nullcontext
        from torch.profiler import ProfilerActivity, profile
        ctx = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) if rank == 0 else nullcontext()
        with ctx as prof:
            for i in range(5):
                step(*pool[i % 4])
            torch.cuda.synchronize()
        if rank == 0:
            rows = sorted(((e.key, e.device_time_total / 5.0, e.count / 5.0) for e in prof.key_averages()
                           if e.device_time_total > 0 and str(getattr(e, "device_type", "")).endswith("CUDA")
                           and not e.key.startswith(("Optimizer.", "ProfilerStep", "aten::", "autograd::", "nccl:", "DistributedDataParallel"))), key=lambda r: -r[1])
            with open(profile_path, "w") as f:
                json.dump({"impl": "torch-gpu", "ms_per_step": ms, "kernels_us_per_step":
                           [{"name": k[:120], "us": round(us, 2), "launches": round(n, 2)} for k, us, n in rows[:160]]},
                          f, indent=1)
        barrier()
    if with_e2e:
        # end to end, the way the reference feeds a GPU: this step's batch comes from host memory
        # (pinned here — the reference's is pageable) and the loss is read back every step
        host = [([t.cpu().pin_memory() for t in d], [tuple(t.cpu().pin_memory() for t in h) for h in tg])
                for d, tg in pool]

        def e2e_step(i):
            d, tg = host[i % 4]
            data = [t.to(dev, non_blocking=True) for t in d]
            target = [tuple(t.to(dev, non_blocking=True) for t in h) for h in tg]
            return step(data, target).item()

        for i in range(3):
            e2e_step(i)
        barrier()
        align_ranks(world, dev)
        e0.record()
        for i in range(steps):
            e2e_step(i)
        e1.record()
        barrier()
        ems = max_over_ranks(e0.elapsed_time(e1)) / steps
        h2d = sum(t.numel() * t.element_size() for t in host[0][0]) + sum(
            t.numel() * t.element_size() for h in host[0][1] for t in h)
        res["e2e"] = {"value": world * B / (ems / 1e3), "unit": "samples/s", "ms_per_step": ems,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4}
    del net, model, opt, pool
    torch.cuda.empty_cache()
    return res


def align_ranks(world, dev):
    """Device-side barrier enqueued right before a start event (world > 1): a 1-element NCCL
    all-reduce completes on every GPU when the LAST rank has enqueued it, so the start events of
    all ranks are recorded within microseconds of one another.  The host barrier before it lets
    the ranks go up to a millisecond apart (8 GPUs: first timed step 1.86 ms against 1.02 for the
    rest, all of it one rank waiting at the first exchange for a peer that started later)."""
    if world > 1:
        import torch
        import torch.distributed as dist
        dist.all_reduce(torch.zeros(1, device=dev))


def main_torch_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    with ClockSampler(local_rank) as clocks:
        res = run_torch_gpu(args, rank, local_rank, world, args.steps, args.warmup, with_e2e=not args.no_e2e,
                            profile_path=args.profile)
    if rank == 0:
        line = {"impl": "torch-gpu", "metric": METRIC, "value": res["value"], "unit": "samples/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
                "config": {"workload": workload_name(args), "global_batch": args.batch * world,
                           "parallelism": "dp%d" % world, "optimizer": res["optimizer"],
                           "grad_allreduce": res["grad_sync"], "precision": res["precision"],
                           "step_issue": res["step"]},
                "e2e": res.get("e2e"), "gpu_launches": 0, "clocks": clocks.summary()}
        emit_line(line)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------

BYTES_PER_PARAM = {  # algorithmic, fp32 master + state, bf16 gradient read, bf16 shadow written
    ("sgd", "bf16"): 2 + 4 + 4 + 4 + 4 + 2, ("sgd", "fp32"): 4 + 4 + 4 + 4 + 4,
    ("adam", "bf16"): 2 + 4 * 3 + 4 * 3 + 2, ("adam", "fp32"): 4 * 4 + 4 * 3,
    ("rmsprop", "bf16"): 2 + 4 * 3 + 4 * 3 + 2, ("rmsprop", "fp32"): 4 * 4 + 4 * 3}


def gpu_numa_node(local_rank):
    """NUMA node the GPU hangs off (sysfs, via its PCI bus id); 0 if unknown."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        with open("/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]) as f:
            return max(int(f.read().strip()), 0)
    except Exception:                                   # noqa: BLE001
        return 0


def shared_global_fields(sample_fields, n_rows, rank, local_rank, world, dev, bf16_fields=()):
    """world > 1: ONE copy of the synthetic dataset per NUMA node of the box.  The lowest rank of
    each node (its threads are bound to the node: first touch lands there) writes every field as
    a file in /dev/shm (a base block of random rows tiled to ``n_rows``, same generator seed on
    every node: the copies are identical; the values are synthetic, the row count and byte volume
    are what the loop sees); every rank maps its node's files and page-locks the mapping
    (cudaHostRegister) so its GPU reads the rows in place over its own PCIe link without crossing
    the socket interconnect."""
    import torch
    import torch.distributed as dist
    tag = os.environ.get("MASTER_PORT", "0")
    node = gpu_numa_node(local_rank)
    nodes = [None] * world
    dist.all_gather_object(nodes, node)
    writer = min(r for r in range(world) if nodes[r] == node) == rank
    out = {}
    paths = {name: "/dev/shm/frl_b200_bench_%s_n%d_%s.bin" % (tag, node, name) for name in sample_fields}
    # fields the transform declares bf16-tolerant are stored in that wire dtype (what the loader
    # would otherwise make of them once per rank: world copies of the global array)
    sample_fields = {k: (v.to(torch.bfloat16) if k in bf16_fields and v.dtype == torch.float32 else v)
                     for k, v in sample_fields.items()}
    if writer:
        try:
            torch.set_num_threads(max(1, min(16, len(os.sched_getaffinity(0)))))
        except AttributeError:
            pass
        g = torch.Generator().manual_seed(7)
        for name, sample in sample_fields.items():
            shape = (n_rows,) + tuple(sample.shape[1:])
            t = torch.from_file(paths[name], shared=True, size=int(torch.tensor(shape).prod()),
                                dtype=sample.dtype).view(shape)
            row_bytes = max(int(sample[0].numel()) * sample.element_size(), 1)
            base = max(1, min(n_rows, 32768, (1 << 29) // row_bytes))      # <= 512 MB of fresh random rows
            if sample.dtype in (torch.float32, torch.bfloat16):
                t[:base].copy_(torch.randn((base,) + shape[1:], generator=g))
            elif sample.dtype == torch.uint8:
                t[:base].copy_(torch.randint(0, 256, (base,) + shape[1:], generator=g, dtype=torch.uint8))
            else:       # integer labels: same range as the sample rows
                hi = int(sample.max().item()) + 1 if sample.numel() else 1
                t[:base].copy_(torch.randint(0, max(hi, 2), (base,) + shape[1:], generator=g, dtype=sample.dtype))
            for lo in range(base, n_rows, base):
                t[lo:lo + base].copy_(t[:min(base, n_rows - lo)])
            del t
    dist.barrier()
    cudart = torch.cuda.cudart()
    for name, sample in sample_fields.items():
        shape = (n_rows,) + tuple(sample.shape[1:])
        t = torch.from_file(paths[name], shared=True, size=int(torch.tensor(shape).prod()),
                            dtype=sample.dtype).view(shape)
        rc = cudart.cudaHostRegister(t.data_ptr(), t.numel() * t.element_size(), 0)
        assert int(rc) == 0, "cudaHostRegister failed: %s" % (rc,)
        assert t.is_pinned()
        out[name] = t
    dist.barrier()
    if writer:
        for path in paths.values():
            os.unlink(path)                   # the mappings keep the memory alive
    return out, len(set(nodes))


def nvls_parity_check(worker, step_fn, world, algo, precision):
    """world > 1, after the timed region: ONE more step from the same weights, optimizer state and
    batch, once through the fused NVLS kernel (K7: in-switch reduce + sharded update + multicast)
    and once through ncclAllReduce + K2 (the un-fused path), eager launches both; reports the
    difference of the resulting fp32 master weights and first optimizer-state vector and asserts
    it is the reduction-order / bf16-rounding bound.  Driver-side evidence that the exchange every
    multi-GPU number ran on computes what NCCL + the plain update computes."""
    import torch
    import torch.distributed as dist
    pipe, opt, arena = worker.pipeline, worker.optimizer, worker.arena
    nv = pipe.nvls
    if nv is None:
        return None
    graphed, worker.graphed = worker.graphed, None
    torch.cuda.synchronize()
    pipe.sync_sharded_state()                      # master + state whole on every rank
    names = list(opt._vec)
    saved = {"master": arena.master.clone(), "lp": None if arena.lp is None else arena.lp.clone(),
             "vec": {k: v.clone() for k, v in opt._vec.items()}, "steps": opt._steps}

    def restore():
        arena.master.copy_(saved["master"])
        if arena.lp is not None:
            arena.lp.copy_(saved["lp"])
        for k, v in saved["vec"].items():
            opt._vec[k].copy_(v)
        opt._steps = saved["steps"]

    def run():
        step_fn()
        torch.cuda.synchronize()
        dist.barrier()
        pipe.sync_sharded_state()
        return arena.master.clone(), (opt._vec[names[0]].clone() if names else None)

    try:
        a_master, a_state = run()                  # K7
        restore()
        pipe.nvls = None
        opt.nvls = None
        b_master, b_state = run()                  # NCCL all-reduce in place + K2
    finally:
        pipe.nvls = nv
        opt.nvls = nv
        worker.graphed = graphed

    def rel(a, b):
        d = (a.double() - b.double())
        return {"max_abs": float(d.abs().max()), "max_rel_to_peak": float(d.abs().max() / b.double().abs().max().clamp_min(1e-30)),
                "rel_l2": float(d.norm() / b.double().norm().clamp_min(1e-30))}

    res = {"what": "one step from identical state and batch: K7 (fused NVLS reduce+update+multicast) "
                   "vs ncclAllReduce + K2, world %d, %s gradients" % (world, "bf16" if precision == "bf16" else "fp32"),
           "master": rel(a_master, b_master),
           # how far that one step moved the weights (so a difference of 0 is not "nothing happened";
           # at world 8 NCCL itself reduces in the NVSwitch and the two paths can agree bit for bit)
           "step_moved_master_rel_l2": float((a_master.double() - saved["master"].double()).norm()
                                             / saved["master"].double().norm().clamp_min(1e-30))}
    if a_state is not None:
        res["state:" + names[0]] = rel(a_state, b_state)
    # bounds: the update moves a weight by lr x (reduced gradient); the two reductions differ by
    # summation order (fp32) or by where the bf16 rounding of the sum happens (bf16 gradients)
    bound_master = 1e-4 if precision == "bf16" else 2e-6
    bound_state = 2e-2 if precision == "bf16" else (1e-5 if algo == "sgd" else 1e-4)
    res["bounds"] = {"master_max_rel_to_peak": bound_master, "state_rel_l2": bound_state}
    ok = res["master"]["max_rel_to_peak"] <= bound_master
    if a_state is not None:
        ok = ok and res["state:" + names[0]]["rel_l2"] <= bound_state
    res["ok"] = bool(ok)
    flag = torch.tensor([0 if ok else 1], device=arena.device)
    dist.all_reduce(flag)
    assert int(flag.item()) == 0, "K7 vs NCCL+K2 parity check failed: %s" % json.dumps(res)
    return res


DUMP_MAX_ELEMS = 1 << 22          # 16 MB of float32 per array: about 34 MB in all for the mlp workload


def dump_outputs(out_dir, result, master):
    """Write what one training step returned to its caller (per-task model outputs, total and
    per-task losses) and the master weights it left, as float32 ``out_dir/<name>.npy``.  An array
    of more than DUMP_MAX_ELEMS elements is replaced by the elements at a fixed seeded sample of
    flat indices (``<name>_sample.npy``), so that two builds can be compared file by file."""
    import re
    import numpy as np
    import torch
    output, total_loss, sub_loss, _ = result
    arrays = {"loss_total": total_loss}
    arrays.update(("loss_" + re.sub(r"[^\w.-]", "_", k), v) for k, v in sub_loss.items())
    arrays.update(("output_%d" % i, o) for i, o in enumerate(output))
    arrays["master_weights"] = master
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach().reshape(-1)
        if t.numel() > DUMP_MAX_ELEMS:
            gen = torch.Generator().manual_seed(0)
            idx = torch.randperm(t.numel(), generator=gen)[:DUMP_MAX_ELEMS].sort().values
            t, name = t[idx.to(t.device)], name + "_sample"
        a = t.float().cpu().numpy()
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= 64 << 20, total
    log("dumped %d arrays (%.1f MB) of the last timed step to %s" % (len(arrays), total / 2 ** 20, out_dir))


def main_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import frl_b200  # noqa: F401
    from frl_b200 import _native, graph_step, synthetic
    from frl_b200.solver import Solver, SolverWorkerArgs, bind_to_gpu_numa_node
    from frl_b200.solver_worker import LossLog
    from frl_b200.types import Device, Precision

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)         # pinned staging buffers on the GPU's NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ns = synthetic.api_namespace("frl_b200")
    t = ns.types
    precision = Precision(args.precision)
    B = args.batch

    torch.manual_seed(0)
    save_dir = "/tmp/frl_b200_bench_%d" % rank
    os.makedirs(save_dir, exist_ok=True)
    problem = build_problem(ns, save_dir, args)
    wargs = SolverWorkerArgs(run_opts=run_opts_for(ns, args.algo, B), problem=problem,
                             save_dir=save_dir, run_device=Device.GPU, node_idx=0, node_count=1,
                             rank=rank, local_rank=local_rank, world_size=world, group_name=None,
                             init_method="env://", precision=precision)
    if args.bucket_mb is not None:
        os.environ["FRL_B200_BUCKET_MB"] = str(args.bucket_mb)
    os.environ["FRL_B200_CUDA_GRAPH"] = "1" if args.graph else "0"
    worker, _, _ = Solver.build_worker(wargs)
    worker.model.train()
    worker.criterion.train()
    arena = worker.arena
    n_tasks = len(worker.criterion.loss_names)
    log("rank %d: arena %d elements, grad dtype %s, buckets %d" % (
        rank, arena.numel, arena.grad_dtype, len(worker.pipeline.buckets)))

    # ---- synthetic batches (generated on the device; seed 1234 + rank) ----
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    POOL = 4
    pool = [synthetic_batch(args, B, gen, dev) for _ in range(POOL)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        tv = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        return tv.item()

    W, K = args.warmup, args.steps
    log_ring = LossLog(n_tasks, W + K + 32, dev)

    def step_resident(i):
        data, target = pool[i % POOL]
        worker.criterion.set_step_sink(log_ring.row(i), log_ring.nan_flag)
        return worker._pass_one_minibatch(i, t.Split.TRAIN, data, target)

    # ======================= leg 1: inputs resident in HBM =======================
    # spin-up: a GPU that sat idle (every GPU but the first on a fresh multi-GPU box) needs tens of
    # milliseconds of load to reach its clocks — longer than W warm-up steps of ~1 ms.  Not a
    # training step: a plain GEMM loop on scratch tensors, before the warm-up steps.
    spin = torch.randn(4096, 4096, device=dev, dtype=torch.bfloat16)
    t_spin = time.perf_counter()
    while time.perf_counter() - t_spin < 0.25:
        for _ in range(20):
            spin = (spin @ spin).clamp_(-1, 1)
        torch.cuda.synchronize()
    del spin
    for i in range(W):
        step_resident(i)
    barrier()
    worker.pipeline.update_events.clear()
    worker.pipeline.record_update_events = True
    launches0 = _native.launch_count() + graph_step.REPLAYED_LAUNCHES
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    with ClockSampler(local_rank) as clocks:
        align_ranks(world, dev)
        marks[0].record()
        host_t0 = time.perf_counter()
        for i in range(K):
            last = step_resident(W + i)
            marks[i + 1].record()
        host_issue_ms = 1e3 * (time.perf_counter() - host_t0) / K     # CPU time to ISSUE a step
        barrier()
    if args.dump_outputs and rank == 0:
        # before any further step: under graph replay the returned tensors are the graph's buffers
        dump_outputs(args.dump_outputs, last, arena.master)
    launches = _native.launch_count() + graph_step.REPLAYED_LAUNCHES - launches0
    worker.pipeline.record_update_events = False
    total_ms = marks[0].elapsed_time(marks[K])
    step_ms = [marks[i].elapsed_time(marks[i + 1]) for i in range(K)]
    total_ms = max_over_ranks(total_ms)
    value = world * B * K / (total_ms / 1e3)
    losses = log_ring.rows[W:W + K, 0]
    assert torch.isfinite(losses).all(), "non-finite loss in the timed region"

    # roofline of the dominant kernel of OUR path: the fused update (K2), timed live by events
    # recorded on the launching stream around every launch inside the timed region.  When the
    # update launches live inside the replayed graph (multi-GPU) they cannot carry timing events,
    # so a few eager steps right after the timed region supply them.
    roofline_from = "events around every update launch inside the timed region"
    if not worker.pipeline.update_events:
        graphed, worker.graphed = worker.graphed, None
        worker.pipeline.record_update_events = True
        for i in range(6):
            step_resident(W + K + i)
        barrier()
        worker.pipeline.record_update_events = False
        worker.graphed = graphed
        # drop the first two (cold) eager steps
        per_step = max(len(worker.pipeline.update_events) // 6, 1)
        worker.pipeline.update_events = worker.pipeline.update_events[2 * per_step:]
        roofline_from = "events around the update launches of 4 eager steps run right after the timed region (in the timed region they are nodes of the replayed CUDA graph)"
    upd = worker.pipeline.update_events
    upd_ms = [e0.elapsed_time(e1) for e0, e1, _, _ in upd]
    upd_elems = sum(hi - lo for _, _, lo, hi in upd)
    bpp = BYTES_PER_PARAM[(args.algo, args.precision)]
    peaks_path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    traffic = None
    tpath = os.path.join(REPO, "profiles", "k2_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("%s_%s" % (args.algo, args.precision))
    nv_link = worker.pipeline.nvls
    kernel_name = "frl::update_kernel (fused grad-bucket + optimizer, K2)"
    nvlink = None
    if nv_link is not None and upd_ms:
        # K7: per bucket element this GPU's HBM serves its gradient copy to the switch (2 B, bf16),
        # receives the new shadow weight (2 B) and streams master + state for its 1/world shard
        state_bytes = bpp - 2 - 2 if args.precision == "bf16" else bpp - 4
        bpp = (4 if args.precision == "bf16" else 8) + state_bytes / world
        kernel_name = ("frl::nvls_update (K7: multimem.ld_reduce + sharded update + multimem.st; "
                       "launch time includes its two cross-GPU barriers)")
        g_b = 2 if args.precision == "bf16" else 4
        link_bytes = upd_elems * g_b * (1.0 + 1.0 / world)          # per direction, per GPU
        nvlink = {"bytes_per_direction_per_launch": link_bytes / len(upd_ms),
                  "achieved": link_bytes / (sum(upd_ms) / 1e3) / 1e9, "peak": 770.0, "unit": "GB/s",
                  "peak_source": "measured peer copy per direction (B200_PROFILING.md); 900 nominal",
                  "note": "NVLink 5 per-direction payload of the fused step: out = own gradient copy "
                          "read by the switch + multicast of the shard's new weights, in = reduced shard "
                          "+ every shard's new weights; this, the barriers and the SMs left over by the "
                          "overlapped backward GEMMs bound K7, not HBM"}
    achieved = bpp * upd_elems / (sum(upd_ms) / 1e3) / 1e9 if upd_ms else None
    roofline = {"bound": "hbm", "kernel": kernel_name,
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "peak_source": peak_src, "bytes_per_param": bpp, "timed_by": roofline_from,
                "elems_per_launch": upd_elems / max(len(upd), 1),
                "avg_launch_ms": (sum(upd_ms) / len(upd_ms)) if upd_ms else None,
                "update_ms_per_step": (sum(upd_ms) / len(upd_ms)) * (arena.numel / (upd_elems / len(upd_ms))) if upd_ms else None}
    if roofline["update_ms_per_step"]:
        roofline["share_of_step"] = roofline["update_ms_per_step"] / (total_ms / K)
    if nvlink is not None:
        roofline["nvlink"] = nvlink
        roofline["traffic"] = None
        roofline["note"] = ("multi-GPU: the update is sharded 1/world per rank and overlapped with "
                            "backward; the single-GPU run carries the HBM roofline of the update kernel (K2)")

    if args.profile:
        # every rank runs the steps (collectives!); only rank 0 records.  Output: a JSON summary of
        # device time per kernel per step (same format as the torch-gpu arm writes) for the
        # kernel-by-kernel attribution of the step-time difference.
        from contextlib import nullcontext
        from torch.profiler import ProfilerActivity, profile
        ctx = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) if rank == 0 else nullcontext()
        with ctx as prof:
            for i in range(5):
                step_resident(W + K + i)
            torch.cuda.synchronize()
        if rank == 0:
            rows = sorted(((e.key, e.device_time_total / 5.0, e.count / 5.0) for e in prof.key_averages()
                           if e.device_time_total > 0 and str(getattr(e, "device_type", "")).endswith("CUDA")
                           and not e.key.startswith(("Optimizer.", "ProfilerStep", "aten::", "autograd::", "nccl:", "DistributedDataParallel"))), key=lambda r: -r[1])
            with open(args.profile, "w") as f:
                json.dump({"impl": "b200", "ms_per_step": total_ms / K, "kernels_us_per_step":
                           [{"name": k[:120], "us": round(us, 2), "launches": round(n, 2)} for k, us, n in rows[:160]]},
                          f, indent=1)
            log(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25))
    barrier()

    # ======================= leg 2: end to end through the public loop =======================
    e2e = None
    if not args.no_e2e:
        # What a user's Solver.solve() runs per epoch: SolverWorker._pass_one_epoch over the
        # Problem's own dataset.  The dataset (fp32) lives in pinned HOST memory behind
        # `problem.datasets`; the loop's DeviceBatchLoader shuffles it with the reference's sampler
        # machinery, moves the rows of the next batches to HBM while the current one trains
        # (FRL_B200_INPUT_PATH: native host gather threads + one DMA per field, or GPU-pulled over
        # PCIe) and runs the transform on the device (frl_preproc_affine -> bf16).  Inside the
        # timed region, every step: H2D of that step's inputs, the step, the loss row landing in
        # pinned host memory (read by the host 2 steps late for the NaN guard), and the loop's
        # bookkeeping — retained batches, per-sample metrics of the Problem's
        # compute_batch_metrics hook read back every metricAmortizationSchedule (10) steps, epoch
        # summary.  One epoch of K steps is timed, after one warm-up epoch over the same loader.
        from frl_b200.device_loader import DeviceBatchLoader
        from frl_b200 import synthetic as syn
        from frl_b200.types import Mode

        from frl_b200.sampler import ScaffoldSampler

        L = K if K <= 128 else K // ((K + 127) // 128)        # steps per epoch
        n_epochs_timed = max(1, K // L)
        # the dataset: L x B samples per rank.  world > 1: ONE global dataset of L x B x world samples
        # in shared host memory, page-locked by every rank, partitioned per epoch by the product's
        # ScaffoldSampler (global randperm seeded by the epoch -> pad -> [rank::world], the
        # reference's bit-exact partition) — every rank gathers ITS rows of the global array.
        host_problem = build_problem(ns, save_dir, args, n_train=L * B if world == 1 else 8, pinned=True,
                                     fast_fields=True, uint8=args.workload != "mlp")
        host_ds = host_problem.datasets[0]
        out_dtype = torch.bfloat16 if precision == Precision.BF16 else torch.float32
        if world > 1:
            tolerant = getattr(host_ds.device_transform, "bf16_wire_fields", ()) if out_dtype == torch.bfloat16 else ()
            # the global dataset lives in /dev/shm: shorten the epoch if the box's tmpfs is small
            row_bytes = sum(t[0].numel() * (2 if (k in tolerant and t.dtype == torch.float32) else t.element_size())
                            for k, t in host_ds.pinned_fields.items())
            st = os.statvfs("/dev/shm")
            fit = int(0.7 * st.f_bavail * st.f_frsize // max(2 * row_bytes * B * world, 1))   # a copy per NUMA node
            if fit < L:
                assert fit >= 4, "/dev/shm too small for a 4-step epoch of the global dataset"
                log("note: /dev/shm holds only %d steps of the global dataset; epoch shortened from %d" % (fit, L))
                L = fit
                n_epochs_timed = max(1, K // L)
            host_ds.pinned_fields, n_copies = shared_global_fields(
                host_ds.pinned_fields, L * B * world, rank, local_rank, world, dev, bf16_fields=tuple(tolerant))
            host_ds._n = L * B * world
        sampler = None
        if world > 1:
            sampler = ScaffoldSampler(host_ds, shuffle_type=t.ShuffleType.RANDPERM, node_idx=0, node_count=1)
        loader = DeviceBatchLoader(host_ds, batch_size=B, device=dev, out_dtype=out_dtype, sampler=sampler)
        assert len(loader) == L, (len(loader), L)
        loaders = {t.Split.TRAIN: loader}
        h2d_bytes = loader.h2d_bytes_per_batch
        worker.cur_epoch = 1
        worker._pass_one_epoch(host_problem, loaders, Mode.TRAIN)        # warm-up epoch (graph capture)
        barrier()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches_e0 = _native.launch_count() + graph_step.REPLAYED_LAUNCHES
        align_ranks(world, dev)
        m0.record()
        for ep in range(n_epochs_timed):
            worker.cur_epoch = 2 + ep
            stats = worker._pass_one_epoch(host_problem, loaders, Mode.TRAIN)
        m1.record()
        barrier()
        e2e_launches = _native.launch_count() + graph_step.REPLAYED_LAUNCHES - launches_e0
        e2e_steps = n_epochs_timed * L
        e2e_ms = max_over_ranks(m0.elapsed_time(m1))
        ep_losses = stats[t.Split.TRAIN].losses
        assert all(v == v for v in ep_losses.values()), "NaN loss in the e2e leg"
        if args.profile and world == 1:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                worker.cur_epoch += 1
                worker._pass_one_epoch(host_problem, loaders, Mode.TRAIN)
                torch.cuda.synchronize()
            rows = sorted(((e.key, e.device_time_total / L, e.count / L) for e in prof.key_averages()
                           if e.device_time_total > 0 and str(getattr(e, "device_type", "")).endswith("CUDA")
                           and not e.key.startswith(("Optimizer.", "ProfilerStep", "aten::", "autograd::", "nccl:", "DistributedDataParallel"))), key=lambda r: -r[1])
            with open(args.profile.replace(".json", "") + "_e2e.json", "w") as f:
                json.dump({"impl": "b200 e2e epoch", "steps": L, "kernels_us_per_step":
                           [{"name": k[:120], "us": round(us, 2), "launches": round(n, 2)} for k, us, n in rows[:160]]},
                          f, indent=1)
        n_metrics = len(stats[t.Split.TRAIN].metrics)
        e2e = {"value": world * B * e2e_steps / (e2e_ms / 1e3), "unit": "samples/s",
               "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": 4 * (1 + n_tasks) + 4 * n_metrics * B,
               "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps, "input_path": loader.path,
               "input_threads": loader.threads, "input_blocks": loader.blocks,
               "input_wire": {k: str(v).replace("torch.", "") for k, v in loader._wire_dtype.items()},
               "gpu_launches": e2e_launches,
               "epoch_losses": {k: float(v) for k, v in ep_losses.items()},
               "sampler": ("ScaffoldSampler (global randperm seeded by the epoch, padded, [rank::world]) over "
                           "one global dataset of %d samples in shared pinned host memory (a copy per NUMA node: %d)" % (L * B * world, n_copies))
                          if world > 1 else "RandomSampler (the reference's single-process loader)",
               "how": "SolverWorker._pass_one_epoch (the loop Solver.solve runs per epoch) over the "
                      "Problem's dataset (%d batches per rank) in pinned host memory, model inputs stored in "
                      "the wire dtype the dataset's transform declares (%s): sampler "
                      "indices -> DeviceBatchLoader moves the rows of the next batches to HBM while "
                      "the current step runs (%s) -> transform + cast on device "
                      "(frl_preproc_affine) -> _pass_one_minibatch (CUDA-graph replay) -> loss row "
                      "written to pinned host memory by the criterion kernel, read 2 steps late; "
                      "includes the loop's retained-batch bookkeeping, the Problem's per-sample "
                      "metric hook every 10 steps and the epoch summary" % (
                          L, ", ".join("%s %s" % (k, str(v).replace("torch.", "")) for k, v in loader._wire_dtype.items()),
                          "native host gather threads into pinned staging + one DMA per field"
                          if loader.path == "host" else
                          "rows pulled over PCIe by frl_gather_rows%s on a copy stream" % (
                              "_tma" if loader.path == "tma" else ""))}

    # ======================= K7 vs NCCL + K2 self-check (N > 1) =======================
    parity = None
    if world > 1 and not args.no_parity_check:
        worker.model.train()
        worker.criterion.train()
        parity = nvls_parity_check(worker, lambda: step_resident(W + K + 100), world, args.algo, args.precision)
        barrier()

    # ======================= stock PyTorch on the same GPU(s) =======================
    torch_base = None
    if not args.no_torch_baseline:
        try:
            torch_base = run_torch_gpu(args, rank, local_rank, world, steps=min(K, 20), warmup=5, with_e2e=False)
            torch_base["speedup_of_value"] = value / torch_base["value"]
        except Exception as e:                      # noqa: BLE001  (a comparison leg must not sink the line)
            log("torch-gpu baseline failed:", repr(e))
            torch_base = {"error": repr(e)[:200]}
        barrier()

    # ======================= CPU baseline (rank 0, N=1) =======================
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = time_cpu_reference(args, args.cpu_batch or WORKLOADS[args.workload]["cpu_sample_batch"],
                                 args.cpu_steps, 1)
        cpu = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}

    nv = worker.pipeline.nvls
    if world == 1:
        grad_sync_desc = "none (1 GPU)"
    elif nv is not None:
        grad_sync_desc = ("fused per-bucket NVLS kernel over NVSwitch multicast (multimem.ld_reduce of the "
                          "bf16 grads + sharded update + multimem.st of the new weights), %d buckets, "
                          "%d CTAs (%d for the last, exposed bucket), barriers %s, tail split %s"
                          % (len(worker.pipeline.buckets), nv.max_blocks, nv.tail_blocks,
                             "as separate 1-CTA launches" if nv.flags & 1 else "in-kernel",
                             "on" if worker.pipeline._row_split else "off"))
    else:
        grad_sync_desc = "NCCL all-reduce in place on bf16 arena buckets + fused update per bucket"
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": total_ms / K, "step_p50_ms": statistics.median(step_ms),
                "step_ms_first5": [round(v, 4) for v in step_ms[:5]], "step_ms_max": max(step_ms),
                "host_issue_ms_per_step": host_issue_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if precision == Precision.BF16 else "f32", "data": "synthetic",
                "config": {"workload": workload_name(args), "global_batch": B * world,
                           "step_issue": "CUDA graph replay" if args.graph else "eager",
                           "spin_up": "0.25 s GEMM loop on scratch tensors before the warm-up steps (clock ramp of an idle GPU; not a training step)",
                           "parallelism": "dp%d" % world,
                           "timed_region": "host barrier + synchronize, then (world > 1) a 1-element NCCL all-reduce "
                                           "enqueued right before the start event so every rank's clock starts "
                                           "together; K steps; event; host barrier + synchronize; max over ranks",
                           "precision": "bf16 forward/backward + bf16 grads, fp32 master weights and "
                                        "optimizer state" if precision == Precision.BF16 else "fp32",
                           "l2": "no flush needed: each step streams the %.1fM-element arena "
                                 "(%.2f GB of update traffic) and 4 rotating input batches, larger than the "
                                 "126 MB L2" % (arena.numel / 1e6, arena.numel * BYTES_PER_PARAM[(args.algo, args.precision)] / 1e9),
                           "grad_allreduce": grad_sync_desc},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
                "torch_gpu_baseline": torch_base, "parity_check": parity,
                "clocks": clocks.summary(), "final_loss": float(losses[-1])}
        emit_line(line)
    if world > 1:
        # Release the captured graphs (they hold NCCL work) before anything NCCL is torn down,
        # line the ranks up, and leave without running communicator destructors: a rank that
        # exits early while another still tears down captured collectives can hang the job.
        import gc
        worker.graphed = None
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its
    version banner on stdout when the box exports NCCL_DEBUG), so file descriptor 1 is pointed at
    stderr for the whole run and the line is written to the saved descriptor at the end."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)

    def emit(line: str) -> None:
        sys.stdout.flush()
        os.write(saved, (line + "\n").encode())

    return emit


EMIT = None


def emit_line(obj) -> None:
    text = json.dumps(obj)
    if EMIT is not None:
        EMIT(text)
    else:
        print(text, flush=True)


def main():
    global EMIT
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl != "reference":
        EMIT = claim_stdout()
    if args.impl == "reference":
        main_reference(args, rank)
        return
    if args.impl == "torch-gpu":
        main_torch_gpu(args, rank, local_rank, world)
        return
    if world != args.gpus:
        log("note: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, world))
    main_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
