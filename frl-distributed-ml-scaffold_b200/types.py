"""Option records and enums of the scaffold plugin API.

Mirrors the public names of the reference's ``types.py`` (reference types.py:36-127) so a
``Problem`` written against the reference constructs the same ``RunOpts``/``OptimOpts`` here.
Field names, order and defaults are the contract; the plotly dependency of the reference's
``SampleSummary.plot`` is dropped (any JSON-serialisable figure dict is accepted).
"""
from enum import Enum
from typing import Any, NamedTuple, Optional

import numpy as np


# --- enums (values are the strings the reference uses on the wire / in logs) ---------------

class ShuffleType(Enum):
    RANDPERM = "randperm"
    PER_NODE_RANDPERM = "per_node_randperm"


class Split(Enum):
    TRAIN = "training"
    TEST = "testing"
    HELDOUT = "heldOut"


class Device(Enum):
    CPU = "cpu"
    GPU = "cuda"


class Mode(Enum):
    EVAL = "eval"
    TRAIN = "train"


class OptAlgorithm(Enum):
    RMSPROP = "rmsprop"
    SGD = "sgd"
    ADAM = "adam"


class LossType(Enum):
    MSE = "mse"
    CrossEntropy = "crossentropy"


class LRSchedulerAlgorithm(Enum):
    DropEpochs = "drop"
    WarmupMultiStepLR = "multistep"


class Precision(Enum):
    """Extension (not in the reference, which is fp32-only): arithmetic of the train step.

    FP32  - parameters, gradients and optimizer state fp32 (reference parity mode, 1e-5 rel).
    BF16  - bf16 shadow weights + bf16 gradients for forward/backward, fp32 master weights and
            optimizer state in the arena, written by the fused update kernel (1e-2 tolerance).
    """
    FP32 = "fp32"
    BF16 = "bf16"


# --- records ---------------------------------------------------------------------------------

class SampleSummary(NamedTuple):
    image: Optional[np.ndarray] = None
    text: Optional[str] = None
    plot: Optional[Any] = None          # plotly Figure or a figure dict
    source: Optional[str] = None


class LRSchedulerOpts(NamedTuple):
    algo: LRSchedulerAlgorithm = LRSchedulerAlgorithm.DropEpochs


class OptimOpts(NamedTuple):
    """Optimizer options (reference types.py:85-93).  How the B200 step consumes them:

    algo          which fused update rule K2/K7 applies (``frl_sgd_momentum`` / ``frl_adam`` /
                  ``frl_rmsprop``); anything else raises ``ValueError`` like the reference
    lr            base rate; the per-epoch scheduler writes the current value into the kernel
                  arguments (or the device-resident ``dyn`` block under CUDA-graph replay)
    lr_scheduler  ``drop`` or ``multistep`` closed forms, stepped once per epoch
    weightDecay   L2-COUPLED decay folded into the gradient read, on every parameter (model and
                  criterion) — this is ``torch.optim``'s ``weight_decay``.  With
                  ``Solver.solve(..., decoupled_weight_decay=True)`` and ADAM it is AdamW's
                  decoupled coefficient instead (p *= 1 - lr*weightDecay before the Adam step;
                  the default 1e-5 stays, torch.optim.AdamW's 1e-2 is not substituted)
    momentum      SGD momentum AND RMSprop momentum (the reference feeds both from this field)
    epsilon       Adam only (RMSprop keeps torch's 1e-8), as in the reference's factory
    amsgrad       Adam: adds the running maximum of the second moment (a third state vector)
    gradientClip  > 0: global-norm clip of the MODEL parameters' gradients (K3 computes the
                  coefficient on the device, K2 applies it); turns the fused NVLS step off
    """
    algo: OptAlgorithm
    lr: float = 0.001
    lr_scheduler: LRSchedulerOpts = LRSchedulerOpts()
    weightDecay: float = 0.00001
    momentum: float = 0.9
    epsilon: float = 1e-8
    amsgrad: bool = False
    gradientClip: float = 0.0


class RunOpts(NamedTuple):
    """Run options (reference types.py:102-121).  Field names, order and defaults are the
    reference's; what each means on the B200 path:

    batchSize                   minibatch PER RANK (weak scaling, as DDP in the reference)
    cpuonly                     must stay False: there is no CPU path, ``Solver.solve`` raises
    nEpochs                     epochs to train; also fixes the LR drop / warm-up milestones
    maxEpochImages              > 0: train on the first N samples of each dataset only
    numThreads                  DataLoader workers of the per-sample input path; the batched
                                device input path (``pinned_fields`` datasets) ignores it
    numIOThreads                accepted for compatibility (storage-layer option)
    metricAmortizationSchedule  every N minibatches the retained outputs/targets are folded
                                into per-sample metrics — on a worker thread here, so the hook's
                                device-to-host read never stalls the step
    initialModelPath            ``state_dict`` to start from (strict in EVAL mode)
    mode                        TRAIN or EVAL (EVAL runs every split forward-only, writes nothing)
    numVisualizedSamples        random + worst-k samples kept per split for the summaries
    singleThreaded              run the single rank in the calling process instead of forking
    outputTTL                   accepted for compatibility (storage-layer option)
    lossLoggingFreq             > 0: log the loss row every N minibatches (a lagged read of the
                                pinned loss log, not a sync)
    debugGrad                   per-task gradient norms at the last shared parameter every 10
                                minibatches; keeps the step on eager launches and stock autograd
    shuffleType                 how ``ScaffoldSampler`` partitions the permutation across ranks
    minibatchTimeoutMs          watchdog: a minibatch longer than this raises ``TimeoutError``
    """
    optim: OptimOpts
    batchSize: int
    cpuonly: bool = False
    nEpochs: int = 75
    maxEpochImages: int = 0
    numThreads: int = 4
    numIOThreads: int = 5
    metricAmortizationSchedule: int = 10
    initialModelPath: Optional[str] = None
    mode: Mode = Mode.TRAIN
    numVisualizedSamples: int = 36
    singleThreaded: bool = False
    outputTTL: int = 0
    lossLoggingFreq: int = 0
    debugGrad: bool = False
    shuffleType: ShuffleType = ShuffleType.RANDPERM
    minibatchTimeoutMs: int = 1000 * 60 * 60


def _fill_namedtuple(cls, args, kwargs):
    merged = dict(cls._field_defaults)
    free = [name for name in cls._fields if name not in kwargs]
    merged.update(zip(free, args))
    merged.update(kwargs)
    return merged


class OptimOptsBase(OptimOpts):
    """Subclassable variant: positional args fill the fields not given by keyword."""

    def __new__(cls, *args, **kwargs):
        return super().__new__(cls, **_fill_namedtuple(cls, args, kwargs))


class RunOptsBase(RunOpts):
    def __new__(cls, *args, **kwargs):
        return super().__new__(cls, **_fill_namedtuple(cls, args, kwargs))
