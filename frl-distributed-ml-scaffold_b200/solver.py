"""``Solver.solve`` — entry point and per-rank bootstrap (reference solver.py:101-837).

Kept from the reference: the ``solve()`` signature and generator protocol, one OS process per
GPU with a one-way pipe back to the parent, per-epoch aggregation (sample-weighted means,
MSE -> RMSE renaming), checkpoint file names and contents, resume from ``.checkpoint.pth``.

Replaced: the per-rank bootstrap no longer wraps the model in ``DistributedDataParallel`` and
``torch.optim``; it builds the flat arena, the fused optimizer and the bucket pipeline
(``arena.py``, ``fused_optim.py``, ``grad_sync.py``).  There is no CPU path: without a CUDA device
(or with ``cpuonly=True``) ``solve`` raises.
"""
import io
import json
import logging
import math
import multiprocessing
import os
import pickle
import traceback
from collections import defaultdict
from contextlib import ExitStack
from multiprocessing.connection import Connection, wait as wait_pipes
from typing import IO, Any, DefaultDict, Dict, Iterator, List, NamedTuple, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .arena import ParamArena
from .criteria import BaseParallelCriterion
from .fused_optim import check_decoupled_weight_decay, create_fused_optimizer
from .grad_sync import BufferBroadcaster, GradBucketPipeline
from .lr_scheduler import DropEpochsScheduler, WarmupMultiStepLR
from .problem import Problem
from .solver_worker import (FractionalPerformanceSummary, SerializableSampleSummary,
                            SolverWorker)
from .types import (Device, LRSchedulerAlgorithm, Mode, Precision, RunOpts, SampleSummary,
                    Split)

logging.basicConfig(level=logging.INFO, format="%(levelname)s (%(process)d) %(message)s")
logger = logging.getLogger(__name__)

CHECKPOINT_NAME = ".checkpoint.pth"
PRECISION_ENV = "FRL_B200_PRECISION"      # "fp32" (default, reference parity) | "bf16"


class SingleSampleSummary(NamedTuple):
    plot: Any
    source: str


class SplitSampleSummaryGroup(NamedTuple):
    image: Optional[bytes]
    text: Optional[str]
    summaries: List[SingleSampleSummary]


class SplitSampleSummary(NamedTuple):
    random: SplitSampleSummaryGroup
    worst: SplitSampleSummaryGroup


class EpochSplitPerformanceSummary(NamedTuple):
    losses: Dict[str, float]
    metrics: Dict[str, float]
    sample_summary: SplitSampleSummary


class PerformanceSummary(NamedTuple):
    epoch: int
    performance: Dict[Split, EpochSplitPerformanceSummary]
    save_dir: str


class Checkpoint(NamedTuple):
    epoch: int
    modelState: Dict[Any, Any]
    optimizerState: Dict[Any, Any]


def _update_rule_name(optimizer) -> str:
    """Name of the update rule in torch's terms, for the one-line path log."""
    name = type(optimizer).__name__.replace("Fused", "")
    if name == "Adam" and optimizer.param_groups[0].get("decoupled_weight_decay", False):
        name = "AdamW"
    return name + (" (amsgrad)" if optimizer.param_groups[0].get("amsgrad", False) else "")


class SolverWorkerArgs(NamedTuple):
    run_opts: RunOpts
    problem: Problem
    save_dir: str
    run_device: Device
    node_idx: int
    node_count: int
    rank: int
    local_rank: int
    world_size: int
    group_name: Optional[str]
    init_method: str
    cache: Any = None
    precision: Precision = Precision.FP32
    save_every: int = 1
    graph_step: Optional[bool] = None      # None: FRL_B200_CUDA_GRAPH (default off)
    decoupled_weight_decay: bool = False   # True with OptAlgorithm.ADAM: AdamW


def _torch_load(f, **kw):
    # checkpoints hold whole pickled modules / optimizer dicts (reference solver.py:604-611)
    return torch.load(f, weights_only=False, **kw)


def _load_model_state(model: nn.Module, model_path: str, strict: bool = True) -> None:
    with open(model_path, "rb") as f:
        new_state = _torch_load(f, map_location="cpu")["state_dict"]
    if strict:
        model.load_state_dict(new_state)
        return
    # partial initialisation: copy what matches in name and shape, report the rest
    own = model.state_dict()
    for name, value in new_state.items():
        if name not in own:
            print("Warning: Parameter named {} is not used by this model.".format(name))
            continue
        value = value.data if isinstance(value, nn.Parameter) else value
        if own[name].size() == value.size():
            own[name].copy_(value)
        else:
            print("Warning: While copying the parameter named {}, whose dimensions in the model "
                  "are {} and whose dimensions in the checkpoint are {}.".format(
                      name, own[name].size(), value.size()))
    for name in own:
        if name not in new_state:
            print("Warning: Parameter named {} in the model is not initialized.".format(name))


def create_lr_scheduler(run_opts: RunOpts, optimizer, checkpoint_epoch=-1):
    """Epoch-granular schedule factory (reference solver.py:191-218)."""
    algo = run_opts.optim.lr_scheduler.algo
    n = run_opts.nEpochs
    if algo == LRSchedulerAlgorithm.DropEpochs:
        drops = [np.floor(n * 0.66667), np.floor(n * 0.9)] if n > 10 else []
        return DropEpochsScheduler(optimizer, drops, last_epoch=checkpoint_epoch)
    if algo == LRSchedulerAlgorithm.WarmupMultiStepLR:
        steps = [np.floor(n * r) for r in (0.33333, 0.66667, 0.9)]
        return WarmupMultiStepLR(optimizer, steps, gamma=0.1, warmup_factor=1.0 / 1000,
                                 warmup_iters=5, warmup_method="linear",
                                 last_epoch=checkpoint_epoch)
    raise ValueError("Unknown optimization algorithm type")


def _save_img(img: Optional[np.ndarray]) -> Optional[bytes]:
    if img is None:
        return None
    import cv2
    ok, png = cv2.imencode(".png", np.flip(img, axis=2))     # RGB -> BGR for OpenCV
    return png.tobytes()


def _aggregate_sample_summaries(results: List[SampleSummary]) -> SplitSampleSummaryGroup:
    images = [s.image for s in results if s.image is not None]
    texts = [s.text for s in results if s.text is not None]
    plots = [SingleSampleSummary(plot=s.plot, source=s.source) for s in results
             if s.plot is not None and s.source is not None]
    return SplitSampleSummaryGroup(
        image=_save_img(np.concatenate(images)) if images else None,
        text="\n".join(texts) if texts else None, summaries=plots)


def _cuda_device_count_without_poisoning_fork() -> int:
    """Device count for the parent process.

    ``torch.cuda.is_available()`` normally goes through ``cudaGetDeviceCount`` which arms torch's
    fork guard: children forked afterwards cannot initialise CUDA ("Cannot re-initialize CUDA in
    forked subprocess") — the stock reference trips over exactly this on current torch
    (reference solver.py:740-747).  The NVML-based check leaves the process fork-safe."""
    os.environ.setdefault("PYTORCH_NVML_BASED_CUDA_CHECK", "1")
    if not torch.cuda.is_available():
        return 0
    return torch.cuda.device_count()


def _fork_is_safe() -> bool:
    """True if a forked child of this process can still initialise CUDA (probed in a throwaway
    child, because the guard's state is only observable after the fork)."""
    if torch.cuda.is_initialized():
        return False
    pid = os.fork()
    if pid == 0:
        code = 1
        try:
            code = 1 if torch._C._cuda_isInBadFork() else 0
        finally:
            os._exit(code)
    _, status = os.waitpid(pid, 0)
    return os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0


def bind_to_gpu_numa_node(local_rank: int) -> bool:
    """Pin this rank's threads to the CPUs nearest its GPU (NVML's ideal affinity), so pinned
    staging buffers are first-touched on the local NUMA node and H2D copies do not cross sockets.
    Best effort: returns False if NVML is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return True
    except Exception as e:                           # noqa: BLE001
        logger.info("NUMA binding skipped: %s", e)
        return False


_NORM_FP32_STATS = {}


def _norm_accepts_fp32_stats(device: torch.device) -> bool:
    """Probe once per device: batch_norm with bf16 input and affine parameters but fp32 running
    statistics (training and eval mode)."""
    key = str(device)
    if key not in _NORM_FP32_STATS:
        try:
            x = torch.randn(4, 3, 2, 2, device=device).to(torch.bfloat16).requires_grad_(True)
            w = torch.ones(3, device=device, dtype=torch.bfloat16, requires_grad=True)
            b = torch.zeros(3, device=device, dtype=torch.bfloat16, requires_grad=True)
            rm, rv = torch.zeros(3, device=device), torch.ones(3, device=device)
            with torch.enable_grad():
                # forward AND backward (torch 2.11's batch_norm backward insists on statistics of
                # the affine parameters' dtype although its forward does not)
                torch.nn.functional.batch_norm(x, rm, rv, w, b, training=True).float().sum().backward()
                torch.nn.functional.batch_norm(x, rm, rv, w, b, training=False).float().sum().backward()
            ok = bool(rm.abs().sum() > 0) and rm.dtype == torch.float32
        except Exception as e:                       # noqa: BLE001
            logger.info("fp32 BatchNorm statistics next to bf16 parameters are not supported here (%s): "
                        "running statistics are kept in bf16", str(e).splitlines()[0])
            ok = False
        _NORM_FP32_STATS[key] = ok
    return _NORM_FP32_STATS[key]


def resolve_precision(explicit: Optional[Precision] = None) -> Precision:
    if explicit is not None:
        return explicit
    return Precision(os.environ.get(PRECISION_ENV, "fp32").lower())


class Solver:
    # ------------------------------------------------------------------------------------------
    # per-rank bootstrap (child process)
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _load_checkpoint(checkpoint_file: IO) -> Checkpoint:
        logger.info("Loading from check point %s", str(checkpoint_file))
        blob = _torch_load(checkpoint_file, map_location="cpu")
        logger.info("Loaded from check point, starting from epoch %d", blob["epoch"])
        return Checkpoint(epoch=blob["epoch"], modelState=blob["state_dict"],
                          optimizerState=blob["optimizer"])

    @staticmethod
    def _init_process_group(args: SolverWorkerArgs, device: torch.device) -> None:
        logger.info("Initializing process group with %s" % args.init_method)
        if torch.distributed.is_initialized():
            return                         # an external launcher (torchrun) already did
        torch.distributed.init_process_group(
            backend="nccl" if device.type == "cuda" else "gloo",
            init_method=args.init_method, world_size=args.world_size, rank=args.rank,
            group_name=args.group_name or "")

    @classmethod
    def build_worker(cls, args: SolverWorkerArgs):
        """Everything `_run_solver_worker` sets up, returned instead of run (bench/tests)."""
        run_opts, problem = args.run_opts, args.problem
        if args.run_device != Device.GPU:
            raise RuntimeError("frl_b200 has no CPU path: a CUDA (sm_100a) device is required")
        torch.cuda.set_device(args.local_rank)
        device = torch.device("cuda", args.local_rank)
        if args.world_size > 1 and os.environ.get("FRL_B200_NUMA_BIND", "1") != "0":
            bind_to_gpu_numa_node(args.local_rank)
        logger.info("Using device %s" % device)

        checkpoint: Optional[Checkpoint] = None
        try:
            with open(os.path.join(args.save_dir, CHECKPOINT_NAME), "rb") as f:
                checkpoint = cls._load_checkpoint(f)
        except FileNotFoundError:
            pass

        # model: build on the host (same RNG stream as the reference), load weights, move
        model = problem.get_model()
        if run_opts.initialModelPath is not None:
            _load_model_state(model, run_opts.initialModelPath,
                              strict=(run_opts.mode == Mode.EVAL))
        elif checkpoint:
            model.load_state_dict(checkpoint.modelState)
        model.to(device)
        criterion: BaseParallelCriterion = problem.get_criterion().to(device)

        distributed = args.world_size > 1
        if distributed:
            cls._init_process_group(args, device)

        # world > 1 without clipping: arena vectors other ranks reach go to symmetric/multicast
        # memory so all-reduce + update + broadcast can be one NVLS kernel per bucket
        symm_alloc = None
        if distributed and not run_opts.optim.gradientClip:
            from .symm import try_make_allocator
            symm_alloc = try_make_allocator(device, args.world_size)
        from .arena_linear import head_layout_groups
        arena = ParamArena(model.parameters(), criterion.parameters(), device=device,
                           precision=args.precision, shared_allocator=symm_alloc,
                           adjacent=head_layout_groups(model))
        if (args.precision == Precision.BF16 and any(b.is_floating_point() for b in model.buffers())
                and not _norm_accepts_fp32_stats(device)):
            # BatchNorm running statistics stay fp32 (what the reference's checkpoints hold: a
            # bf16 EMA with momentum 0.1 stalls on small deltas); only if this torch build
            # refuses bf16 activations/affine parameters next to fp32 statistics are the buffers
            # cast — and upcast again on export (arena.exported)
            for buf in model.buffers():
                if buf.is_floating_point():
                    buf.data = buf.data.to(torch.bfloat16)
        optimizer = create_fused_optimizer(arena, run_opts.optim,
                                           decoupled_weight_decay=args.decoupled_weight_decay)
        if checkpoint:
            optimizer.load_state_dict(checkpoint.optimizerState)
        nvls_link = None
        if symm_alloc is not None:
            from .symm import make_link
            # grid of the fused NVLS step: each rank streams 1/world of a bucket, and every CTA it
            # parks on an SM while backward runs costs the cluster-scheduled GEMMs a wave, so the
            # grid shrinks with the world size.  Measured, ms/step with 24 MiB buckets:
            #   8 x B200: 16 CTAs 1.12 | 32: 1.17 | 74: 1.25 | 148: 1.40
            #   4 x B200:  8 CTAs 1.42 | 16: 1.16 | 37: 1.17 | 74: 1.25
            #   2 x B200: 32 CTAs 1.48 | 74: 1.26 | 148: 1.31   (half of every bucket per rank)
            default_blocks = 74 if args.world_size <= 2 else 16
            # the launch for the bucket that becomes ready last runs alone (backward has ended), so it
            # gets a wider grid: 4 x B200, 16 -> 64 CTAs for that launch only: 1.109 -> 1.074 ms/step
            default_tail = 64 if args.world_size >= 4 else 0
            nvls_link = make_link(symm_alloc, arena.grad,
                                  arena.lp if arena.lp is not None else arena.master,
                                  max_blocks=int(os.environ.get("FRL_B200_NVLS_BLOCKS", default_blocks)),
                                  tail_blocks=int(os.environ.get("FRL_B200_NVLS_TAIL_BLOCKS", default_tail)))
        pipeline = GradBucketPipeline(
            arena, optimizer, world_size=args.world_size, clip_norm=run_opts.optim.gradientClip,
            nvls_link=nvls_link,
            bucket_cap_mb=float(os.environ.get("FRL_B200_BUCKET_MB",
                                               "24" if nvls_link is not None else "48")),
            first_bucket_mb=None,
            eager_update=os.environ.get("FRL_B200_EAGER_UPDATE",
                                        "1" if args.world_size > 1 else "0") != "0")
        # GradNorm differentiates through the layers' backward (create_graph=True) and debugGrad
        # calls autograd.grad on them: those runs keep the stock nn.Linear autograd path
        from .criteria import GradNormWeightedCriterion
        if (os.environ.get("FRL_B200_DIRECT_GRADS", "1") != "0" and not run_opts.debugGrad
                and not isinstance(criterion, GradNormWeightedCriterion)):
            pipeline.patch_linears(model)
        buffers = None
        if distributed:
            pipeline.broadcast_parameters(src=0)
            buffers = BufferBroadcaster(model, world_size=args.world_size)
            buffers.sync()
        worker = SolverWorker(model, criterion, optimizer, device=device, run_opts=run_opts,
                              cache=args.cache, local_rank=args.local_rank,
                              node_idx=args.node_idx, node_count=args.node_count,
                              pipeline=pipeline, buffers=buffers, precision=args.precision,
                              serialize_state=(args.local_rank == 0),
                              graph_step=(args.graph_step if args.graph_step is not None
                                          else os.environ.get("FRL_B200_CUDA_GRAPH", "0") == "1"))
        worker.save_every = args.save_every
        if args.rank == 0:
            # one line per run: which of the alternative paths this configuration took
            logger.info(
                "frl_b200 step: precision %s | update rule %s | step issue %s | gradient exchange %s | "
                "update %s | Linear layers with arena-born gradients %d (%d fused with their ReLU) | "
                "other gradients %s",
                args.precision.value, _update_rule_name(optimizer),
                "CUDA-graph replay after 2 eager steps" if worker.graphed is not None else "eager launches",
                ("fused NVLS kernel per bucket (K7), %d buckets" % len(pipeline.buckets)) if pipeline.nvls is not None
                else ("ncclAllReduce in place + K2 per bucket, %d buckets" % len(pipeline.buckets)) if distributed
                else "none (1 GPU)",
                "per bucket on the side stream" if pipeline.eager else "one tail launch",
                len(pipeline.linear_sites), sum(s.relu is not None for s in pipeline.linear_sites),
                "read in place through segment tables (K2-mt / one flatten launch per bucket)"
                if pipeline.mt_enabled else "copied into the arena per tensor")
        scheduler = create_lr_scheduler(run_opts, worker.optimizer,
                                        checkpoint.epoch if checkpoint else -1)
        return worker, scheduler, checkpoint

    @classmethod
    def _run_solver_worker(cls, args: SolverWorkerArgs) -> Iterator[FractionalPerformanceSummary]:
        """One of ``world_size`` instances, each training on its share of every epoch."""
        worker, scheduler, checkpoint = cls.build_worker(args)
        run_opts = args.run_opts
        if run_opts.mode == Mode.TRAIN:
            yield from worker.train(args.problem,
                                    startEpoch=checkpoint.epoch if checkpoint else 0,
                                    nEpochs=run_opts.nEpochs, batchSize=run_opts.batchSize,
                                    scheduler=scheduler)
        elif run_opts.mode == Mode.EVAL:
            yield from worker.eval(args.problem, batchSize=run_opts.batchSize)
        else:
            raise ValueError("unknown mode")

    @classmethod
    def _solver_worker_process(cls, solver_worker_args: SolverWorkerArgs,
                               comms_connection: Connection, cleanup_flag) -> None:
        """Child main: stream pickled per-epoch results, ``None`` on clean exit, the exception
        object on failure; then hold the pipe open until the parent has drained it."""
        root = logging.getLogger()
        root.setLevel(logging.DEBUG)
        try:
            for result in cls._run_solver_worker(solver_worker_args):
                comms_connection.send_bytes(pickle.dumps(result, protocol=pickle.HIGHEST_PROTOCOL))
            comms_connection.send(None)
        except Exception as e:
            logger.error(str(e))
            for line in traceback.format_exc().splitlines(False):
                logger.error(line)
            try:
                comms_connection.send(e)
            except Exception:
                comms_connection.send(RuntimeError(repr(e)))
            raise
        finally:
            cleanup_flag.wait()

    # ------------------------------------------------------------------------------------------
    # parent side: aggregation
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _deserialize_sample_summaries(items: Sequence[SerializableSampleSummary]
                                      ) -> List[SampleSummary]:
        return [SampleSummary(image=s.image, text=s.text,
                              plot=json.loads(s.plot) if s.plot else None, source=s.source)
                for s in items]

    @classmethod
    def _aggregate_fractional_results(cls, run_opts: RunOpts, problem: Problem,
                                      fractional_results: List[FractionalPerformanceSummary]
                                      ) -> Dict[Split, EpochSplitPerformanceSummary]:
        splits = [d.data_type for d in problem.datasets]
        metric_sum = {s: defaultdict(float) for s in splits}
        loss_sum = {s: defaultdict(float) for s in splits}
        n_samples = {s: 0 for s in splits}
        picked = {s: [] for s in splits}
        worst = {s: [] for s in splits}
        for frac in fractional_results:
            for split, perf in frac.performance.items():
                for k, v in perf.metrics.items():
                    metric_sum[split][k] += v * perf.nSamples
                for k, v in perf.losses.items():
                    loss_sum[split][k] += v * perf.nSamples
                n_samples[split] += perf.nSamples
                picked[split] += cls._deserialize_sample_summaries(perf.samples)
                worst[split] += cls._deserialize_sample_summaries(perf.worstSamples)

        def finish_metrics(split: Split) -> Dict[str, float]:
            # sample-weighted MSE aggregates correctly but reads badly: report RMSE instead
            out: DefaultDict[str, float] = defaultdict(float)
            for name, total in metric_sum[split].items():
                value = total / n_samples[split]
                assert name.find("RMSE") == -1
                if "MSE" in name:
                    head, _, tail = name.rpartition("MSE")
                    out[head + "RMSE" + tail] = math.sqrt(value) if value > 0 else value
                else:
                    out[name] = value
            return out

        return {split: EpochSplitPerformanceSummary(
                    losses={k: v / n_samples[split] for k, v in loss_sum[split].items()},
                    metrics=finish_metrics(split),
                    sample_summary=SplitSampleSummary(
                        random=_aggregate_sample_summaries(picked[split]),
                        worst=_aggregate_sample_summaries(worst[split])))
                for split in splits}

    # ------------------------------------------------------------------------------------------
    # parent side: files
    # ------------------------------------------------------------------------------------------
    @classmethod
    def _save_epoch_summary(cls, epoch: int, save_dir: str,
                            epoch_stats: Dict[Split, EpochSplitPerformanceSummary]) -> None:
        for split, summary in epoch_stats.items():
            for group_name, group in (("random", summary.sample_summary.random),
                                      ("worst", summary.sample_summary.worst)):
                stem = os.path.join(save_dir, ".%s_%s_%04d" % (split.value, group_name, epoch))
                if group.image is not None:
                    with open(stem + ".png", "wb") as f:
                        f.write(group.image)
                if group.text is not None:
                    with open(stem + ".txt", "wb") as f:
                        f.write(group.text.encode("utf-8"))

    @classmethod
    def _save_checkpoint(cls, epoch: int, save_dir: str, run_opts: RunOpts, problem: Problem,
                         fractional_results: List[FractionalPerformanceSummary],
                         base_filename: str) -> None:
        # replicas are identical after every step, so one rank's state stands for all; the
        # rank with local_rank 0 is the one that serialised it
        donors = [r for r in fractional_results if r.modelBuffer]
        if not donors:
            raise RuntimeError("no worker serialised its model state")
        donor = donors[0]
        test_io = None
        for split in (Split.HELDOUT, Split.TEST, Split.TRAIN):
            if split in donor.performance:
                test_io = donor.performance[split].testIO
                break
        if test_io is None:
            raise RuntimeError("No splits found")
        test_input = [torch.stack([s.data[i] for s in test_io]) for i in range(len(test_io[0].data))]
        test_output = [torch.stack([s.output[i] for s in test_io])
                       for i in range(len(test_io[0].output))]
        model = _torch_load(io.BytesIO(donor.modelBuffer), map_location="cpu")
        optimizer_state = _torch_load(io.BytesIO(donor.optimizerStateBuffer), map_location="cpu")

        logger.info("==> saving checkpoint to %s", str(save_dir))
        stem = os.path.join(save_dir, base_filename)
        with ExitStack() as stack:
            f_ckpt = stack.enter_context(open(stem, "wb"))
            f_model = stack.enter_context(open(stem + ".model", "wb"))
            f_data = stack.enter_context(open(stem + ".test_data", "wb"))
            f_anno = stack.enter_context(open(stem + ".annotate_param", "wb"))
            torch.save({"epoch": epoch, "optimizer": optimizer_state,
                        "state_dict": model.state_dict()}, f_ckpt)
            torch.save(model, f_model)       # whole module: loadable without the class layout
            torch.save({"test_input": test_input, "test_output": test_output}, f_data)
            torch.save(problem.anno_param._asdict() if problem.anno_param else {}, f_anno)

    # ------------------------------------------------------------------------------------------
    # parent side: collecting per-epoch results from the ranks
    # ------------------------------------------------------------------------------------------
    @classmethod
    def _collect_direct_fractional_results(cls, args: SolverWorkerArgs
                                           ) -> Iterator[List[FractionalPerformanceSummary]]:
        for res in cls._run_solver_worker(args):
            yield [res]

    @classmethod
    def _collect_process_fractional_results(cls, processes, parent_pipes: List[Connection],
                                            cleanup_flag
                                            ) -> Iterator[List[FractionalPerformanceSummary]]:
        pending: DefaultDict[int, List[FractionalPerformanceSummary]] = defaultdict(list)
        finished: List[Connection] = []
        try:
            while len(finished) < len(processes):
                for pipe in wait_pipes(parent_pipes, 5):
                    try:
                        msg = pipe.recv()
                    except EOFError:
                        if pipe not in finished:
                            raise Exception("Child process failed to exit cleanly.")
                        logger.info("Worker process has exited")
                        continue
                    if msg is None:
                        logger.info("Worker process ready to exit")
                        finished.append(pipe)
                    elif isinstance(msg, Exception):
                        logger.info("Received exception from child process")
                        raise msg
                    else:
                        pending[msg.epoch].append(msg)
                        if len(pending[msg.epoch]) == len(processes):
                            yield pending.pop(msg.epoch)
        except Exception:
            logger.exception("Unexpected error in solve")
            cleanup_flag.set()
            logger.info("Sending SIGTERM to all child processes.")
            for p in processes:
                logger.info("Killing process with pid " + str(p.pid))
                p.terminate()
            raise
        finally:
            cleanup_flag.set()
            logger.info("Joining worker processes")
            for p in processes:
                p.join()

    # ------------------------------------------------------------------------------------------
    # entry point
    # ------------------------------------------------------------------------------------------
    @classmethod
    def solve(cls, run_opts: RunOpts, problem: Problem, *, group_name: Optional[str],
              init_method: str, node_idx: int = 0, node_count: int = 1, memory_quota: int = 0,
              precision: Optional[Precision] = None, graph: Optional[bool] = None,
              decoupled_weight_decay: bool = False) -> Iterator[PerformanceSummary]:
        """The reference's entry point (solver.py:728-739) plus three keyword-only extensions:

        ``precision``  ``Precision.FP32`` (default; parity with the reference's arithmetic) or
                       ``Precision.BF16`` (bf16 forward/backward/gradients, fp32 master weights and
                       optimizer state — the benchmarked configuration).  None: FRL_B200_PRECISION.
        ``graph``      True: replay the training step from a CUDA graph once a batch signature
                       has run 2 eager steps (the Problem's forward must be capturable: static
                       shapes, no host syncs; a failed capture falls back to eager launches).
                       None: FRL_B200_CUDA_GRAPH (default off).
        ``decoupled_weight_decay``  True with ``OptimOpts(algo=OptAlgorithm.ADAM)``: AdamW
                       (``torch.optim.AdamW``; ``OptimOpts.weightDecay`` is the decoupled
                       coefficient, ``epsilon``/``amsgrad`` as for Adam).  With SGD or RMSprop it
                       raises ``ValueError`` before any rank starts.  False (default): Adam's
                       L2-coupled decay, as in the reference.
        """
        check_decoupled_weight_decay(run_opts.optim, decoupled_weight_decay)
        n_visible = 0 if run_opts.cpuonly else _cuda_device_count_without_poisoning_fork()
        if n_visible == 0:
            raise RuntimeError(
                "frl_b200 runs the training step on B200 GPUs only (cpuonly=%s, visible CUDA "
                "devices=%d); there is no CPU path" % (run_opts.cpuonly, n_visible))
        run_device = Device.GPU
        if run_opts.singleThreaded:
            device_count, world_size = 1, 1
        else:
            device_count = n_visible
            world_size = device_count * node_count
        logger.info("World size %d, device count %d" % (world_size, device_count))
        num_workers = min(device_count, world_size)

        save_dir = problem.save_dir + (str(node_idx) if node_count > 1 else "")
        os.makedirs(save_dir, exist_ok=True)
        assert len(problem.datasets) > 0, "datasets cannot be empty"
        # big datasets checkpoint every epoch, small ones every fifth
        save_every = 1 if len(problem.datasets[0]) > 300_000 else 5
        prec = resolve_precision(precision)

        logger.info("Parent process has pid " + str(os.getpid()))
        # fork keeps un-picklable Problems working (as in the reference) but is only safe while
        # this process holds no CUDA context
        use_fork = run_opts.singleThreaded or _fork_is_safe()
        if not use_fork:
            logger.info("CUDA already touched in the parent: ranks are spawned (Problem must pickle)")
        ctx = multiprocessing.get_context("fork" if use_fork else "spawn")
        cleanup_flag = ctx.Event()
        processes, parent_pipes = [], []
        args: Optional[SolverWorkerArgs] = None
        for local_rank in range(num_workers):
            args = SolverWorkerArgs(
                run_opts=run_opts, problem=problem, save_dir=save_dir, run_device=run_device,
                node_idx=node_idx, node_count=node_count,
                rank=node_idx * device_count + local_rank, local_rank=local_rank,
                world_size=world_size, group_name=group_name, init_method=init_method,
                cache=None, precision=prec, save_every=save_every, graph_step=graph,
                decoupled_weight_decay=decoupled_weight_decay)
            if not run_opts.singleThreaded:
                parent_conn, child_conn = ctx.Pipe(duplex=False)
                proc = ctx.Process(target=cls._solver_worker_process,
                                   kwargs={"solver_worker_args": args,
                                           "comms_connection": child_conn,
                                           "cleanup_flag": cleanup_flag})
                proc.start()
                parent_pipes.append(parent_conn)
                processes.append(proc)
                logger.info("Started worker with rank: %d pid: %d", local_rank, proc.pid)
        assert args is not None
        if run_opts.singleThreaded:
            assert num_workers == 1, "Single threaded run cannot use multiple workers"
            results = cls._collect_direct_fractional_results(args)
        else:
            results = cls._collect_process_fractional_results(processes, parent_pipes, cleanup_flag)

        for res in results:
            epoch = res[0].epoch
            epoch_stats = cls._aggregate_fractional_results(run_opts, problem, res)
            if run_opts.mode == Mode.TRAIN:
                final = epoch == run_opts.nEpochs
                if epoch % save_every == 0 or final:
                    cls._save_epoch_summary(epoch, save_dir, epoch_stats)
                    cls._save_checkpoint(epoch, save_dir, run_opts, problem, res,
                                         "final_model.pth" if final else CHECKPOINT_NAME)
            yield PerformanceSummary(epoch=epoch, performance=epoch_stats, save_dir=str(save_dir))
