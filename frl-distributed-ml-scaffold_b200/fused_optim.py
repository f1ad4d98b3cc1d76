"""Arena optimizers: ``torch.optim``-compatible front, one fused kernel launch per bucket behind.

``create_fused_optimizer`` is the B200 counterpart of the reference's ``_create_optimizer``
(reference solver.py:162-188): same three algorithms, same hyper-parameter mapping
(``OptimOpts.momentum`` feeds SGD *and* RMSprop, ``epsilon``/``amsgrad`` feed Adam, weight decay
is L2-coupled and applies to every parameter).  One extension: ``decoupled_weight_decay=True``
turns Adam into AdamW (``torch.optim.AdamW``), still decaying every parameter.
``state_dict()`` / ``load_state_dict()`` speak torch's per-parameter format so the reference's
``.checkpoint.pth`` files stay interchangeable (and an AdamW run's load into ``torch.optim.AdamW``).

Known limitation: the step count (Adam's bias corrections) is ONE number for the whole arena.
``torch.optim`` keeps one per parameter and does not advance it for a parameter whose gradient
is ``None`` in a step; here a parameter that misses gradients for some steps (world size 1 only:
with several ranks a missing gradient is DDP's error, as in the reference) keeps being corrected
with the global count, ``state_dict()`` writes that count for every parameter and
``load_state_dict()`` takes the maximum over the loaded entries.  Models whose parameters all
receive a gradient every step — every configuration of BASELINE.json — are unaffected.
"""
from typing import Any, Dict, List, Optional, Tuple

import torch

from . import _native
from .arena import ParamArena
from .types import OptAlgorithm, OptimOpts

# Kernel entry points; tests exercising host logic on CPU swap this for an oracle-backed double.
KERNELS = _native


class FusedArenaOptimizer(torch.optim.Optimizer):
    """Base: owns the fp32 state vectors (same layout as the arena) and the step counter."""

    STATE_NAMES: Tuple[str, ...] = ()

    def __init__(self, arena: ParamArena, defaults: Dict[str, Any]) -> None:
        self.arena = arena
        params = arena.all_params
        if not params:
            raise ValueError("optimizer got an empty parameter list")
        super().__init__(params, defaults)
        self._vec: Dict[str, torch.Tensor] = {}
        self._steps = 0                # completed optimizer steps
        self._in_step = False
        # device-resident per-step scalars (lr, Adam bias corrections): set when the step is
        # replayed from a CUDA graph, where by-value kernel arguments are frozen at capture
        self._dyn: Optional[torch.Tensor] = None
        self._dyn_last: Optional[Tuple[float, ...]] = None
        # fused NVLS step (world > 1): set by the pipeline; each rank then updates only its
        # 1/world shard of every bucket (master + state), the weights arrive by multicast
        self.nvls = None

    # -- device-resident scalars -----------------------------------------------------------------
    def _dyn_values(self) -> Tuple[float, ...]:
        """Scalars of the NEXT step (``_steps + 1``) in the layout the kernel's ``dyn`` expects."""
        return (float(self.hyper["lr"]),)

    def enable_dynamic_scalars(self) -> None:
        if self._dyn is None:
            self._dyn = torch.zeros(4, dtype=torch.float32, device=self.arena.device)
            self._dyn_last = None
        self.refresh_dynamic_scalars()

    _DYN_RING = 16        # pinned staging rows; the host never runs this many steps ahead

    def refresh_dynamic_scalars(self) -> None:
        """Upload the scalars if they changed: 16 bytes from a ring of pinned rows, so the copy is
        truly asynchronous (a pageable source makes the driver synchronise the stream first,
        which serialises the host's work for step k+1 with the device's work for step k —
        measured on Adam, whose bias corrections change every step: 2.4 vs 1.7 ms/step)."""
        if self._dyn is None:
            return
        vals = self._dyn_values()
        if vals != self._dyn_last:
            if self._dyn.is_cuda:
                if getattr(self, "_dyn_host", None) is None:
                    self._dyn_host = torch.zeros(self._DYN_RING, 4, dtype=torch.float32, pin_memory=True)
                    self._dyn_slot = 0
                row = self._dyn_host[self._dyn_slot % self._DYN_RING]
                self._dyn_slot += 1
                for i, v in enumerate(vals):
                    row[i] = v
                self._dyn.copy_(row, non_blocking=True)
            else:
                self._dyn.copy_(torch.tensor(list(vals) + [0.0] * (4 - len(vals)), dtype=torch.float32))
            self._dyn_last = vals

    # -- state vectors ---------------------------------------------------------------------------
    def _state(self, name: str) -> torch.Tensor:
        v = self._vec.get(name)
        if v is None:
            v = self._vec[name] = self.arena.new_state()
        return v

    @property
    def hyper(self) -> Dict[str, Any]:
        return self.param_groups[0]

    # -- stepping --------------------------------------------------------------------------------
    def begin_step(self) -> None:
        """Open step ``_steps + 1``; per-bucket ``apply_range`` calls share its number."""
        self._in_step = True
        # an EAGER step after a graph was captured (ragged last batch, a second batch signature):
        # the kernels still read the device-resident scalars, so they must be this step's.  Never
        # inside a capture: the copy would be frozen into the graph and undo the per-replay upload.
        if self._dyn is not None and not (self._dyn.is_cuda and torch.cuda.is_current_stream_capturing()):
            self.refresh_dynamic_scalars()

    def end_step(self) -> None:
        self._steps += 1
        self._in_step = False

    def apply_range(self, lo: int, hi: int, *, grad_scale: float = 1.0,
                    clip_coef_dev: Optional[torch.Tensor] = None) -> None:
        """Update arena elements ``[lo, hi)``.  ``clip_coef_dev`` (a device scalar written by
        the norm kernel) multiplies model-parameter gradients only — the reference clips
        ``model.parameters()`` and leaves criterion parameters alone
        (reference solver_worker.py:588-591)."""
        if hi <= lo:
            return
        split = self.arena.model_end
        if clip_coef_dev is not None and lo < split < hi:
            self._launch(lo, split, grad_scale, clip_coef_dev)
            self._launch(split, hi, grad_scale, None)
        else:
            self._launch(lo, hi, grad_scale, clip_coef_dev if lo < split else None)

    def _launch(self, lo: int, hi: int, grad_scale: float, coef) -> None:
        raise NotImplementedError

    def apply_table(self, table, *, grad_scale: float = 1.0) -> None:
        """Update every arena slot listed in ``table`` (a ``multi_tensor.GradSegTable`` whose device
        copy is current), reading each gradient where the table says it lies (K2-mt)."""
        if table.n_segs:
            self._launch_mt(table, grad_scale)

    def _launch_mt(self, table, grad_scale: float) -> None:
        raise NotImplementedError

    # -- fused all-reduce + update + broadcast (K7) ------------------------------------------------
    def apply_range_nvls(self, lo: int, hi: int, *, grad_scale: float) -> None:
        if hi > lo:
            split = bool(self.nvls.flags & KERNELS.NVLS_EXTERNAL_SYNC)
            if split:
                KERNELS.nvls_barrier(self.nvls, 0)     # every rank's bucket gradients are written
            self._launch_nvls(lo, hi, grad_scale)
            if split:
                KERNELS.nvls_barrier(self.nvls, 1)     # every replica has every shard

    def _launch_nvls(self, lo: int, hi: int, grad_scale: float) -> None:
        raise NotImplementedError

    def _nvls_ptrs(self, lo: int):
        k = self.nvls
        return k.mc_grad + lo * k.grad_esz, k.mc_out + lo * k.out_esz

    def shard_of(self, lo: int, hi: int) -> Tuple[int, int]:
        """Element range of bucket ``[lo, hi)`` this rank owns under the fused NVLS step (same
        formula as csrc/nvls.cu)."""
        k = self.nvls
        n = hi - lo
        per = ((n + k.world - 1) // k.world + 7) // 8 * 8
        a = min(lo + k.rank * per, hi)
        return a, min(a + per, hi)

    @torch.no_grad()
    def step(self, closure=None, *, grad_scale: float = 1.0,
             clip_coef_dev: Optional[torch.Tensor] = None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self.begin_step()
        self.apply_range(0, self.arena.numel, grad_scale=grad_scale, clip_coef_dev=clip_coef_dev)
        self.end_step()
        return loss

    def zero_grad(self, set_to_none: bool = True) -> None:
        # Gradients are overwritten (first touch is a store, not an accumulate), so there is
        # nothing to clear in the arena; dropping stray .grad tensors keeps autograd stealing.
        for p in self.arena.all_params:
            p.grad = None

    # -- views used by the launchers -------------------------------------------------------------
    def _slices(self, lo: int, hi: int):
        a = self.arena
        lp = a.lp[lo:hi] if (a.lp is not None and lo < a.model_end) else None
        return a.master[lo:hi], a.grad[lo:hi], lp

    # -- torch-format (de)serialisation ----------------------------------------------------------
    def _per_param_extra(self) -> Dict[str, Any]:
        return {}

    def state_dict(self) -> Dict[str, Any]:
        state: Dict[int, Dict[str, Any]] = {}
        if self._steps > 0:
            for s in sorted(self.arena.slots, key=lambda s: s.index):     # torch's key order
                entry = dict(self._per_param_extra())
                for torch_name, vec_name in self.STATE_NAMES:
                    if vec_name in self._vec:
                        entry[torch_name] = self._vec[vec_name][s.offset:s.end].view(s.shape).clone()
                state[s.index] = entry
        groups = []
        for g in self.param_groups:
            packed = {k: v for k, v in g.items() if k != "params"}
            packed["params"] = list(range(len(g["params"])))
            groups.append(packed)
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, state_dict: Dict[str, Any]) -> None:
        groups = state_dict["param_groups"]
        if len(groups) != 1 or len(groups[0]["params"]) != len(self.arena.all_params):
            raise ValueError("loaded state dict has a different number of parameters/groups")
        for k, v in groups[0].items():
            if k != "params":
                self.param_groups[0][k] = v
        by_index = {s.index: s for s in self.arena.slots}
        steps = 0
        for idx, entry in state_dict["state"].items():
            s = by_index.get(int(idx))
            if s is None:
                continue
            for torch_name, vec_name in self.STATE_NAMES:
                if torch_name in entry and entry[torch_name] is not None:
                    self._state(vec_name)[s.offset:s.end].view(s.shape).copy_(entry[torch_name])
            if "step" in entry:
                steps = max(steps, int(float(entry["step"])))
            elif entry:
                steps = max(steps, 1)
        self._steps = steps


class FusedSGD(FusedArenaOptimizer):
    STATE_NAMES = (("momentum_buffer", "momentum_buffer"),)

    def __init__(self, arena, lr, momentum=0.0, dampening=0.0, weight_decay=0.0):
        super().__init__(arena, dict(lr=lr, momentum=momentum, dampening=dampening,
                                     weight_decay=weight_decay, nesterov=False, maximize=False,
                                     foreach=None, differentiable=False, fused=None))

    def _launch(self, lo, hi, grad_scale, coef):
        h = self.hyper
        p, g, lp = self._slices(lo, hi)
        mu = float(h["momentum"])
        buf = self._state("momentum_buffer")[lo:hi] if mu != 0.0 else None
        KERNELS.sgd_momentum(p, g, buf, lp, hi - lo, lr=float(h["lr"]), mu=mu,
                             dampening=float(h["dampening"]), wd=float(h["weight_decay"]),
                             grad_scale=grad_scale, grad_scale_dev=coef,
                             first_step=(self._steps == 0), dyn=self._dyn)

    def _launch_mt(self, table, grad_scale):
        h = self.hyper
        mu = float(h["momentum"])
        KERNELS.sgd_momentum_mt(self.arena.master, self._state("momentum_buffer") if mu != 0.0 else None,
                                self.arena.lp, table, lr=float(h["lr"]), mu=mu,
                                dampening=float(h["dampening"]), wd=float(h["weight_decay"]),
                                grad_scale=grad_scale, first_step=(self._steps == 0), dyn=self._dyn)

    def _launch_nvls(self, lo, hi, grad_scale):
        h = self.hyper
        mu = float(h["momentum"])
        mc_g, mc_out = self._nvls_ptrs(lo)
        buf = self._state("momentum_buffer")[lo:hi] if mu != 0.0 else None
        KERNELS.nvls_sgd(self.arena.master[lo:hi], buf, mc_g, mc_out, hi - lo, self.nvls,
                         lr=float(h["lr"]), mu=mu, dampening=float(h["dampening"]),
                         wd=float(h["weight_decay"]), grad_scale=grad_scale,
                         first_step=(self._steps == 0),
                         g_dtype=KERNELS.dtype_code(self.arena.grad.dtype), dyn=self._dyn)


class FusedAdam(FusedArenaOptimizer):
    STATE_NAMES = (("exp_avg", "exp_avg"), ("exp_avg_sq", "exp_avg_sq"),
                   ("max_exp_avg_sq", "max_exp_avg_sq"))

    def __init__(self, arena, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, *,
                 decoupled_weight_decay=False):
        super().__init__(arena, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay,
                                     amsgrad=amsgrad, maximize=False, foreach=None,
                                     capturable=False, differentiable=False, fused=None,
                                     decoupled_weight_decay=bool(decoupled_weight_decay)))

    @property
    def decoupled(self) -> bool:
        """torch's ``decoupled_weight_decay``: read from the param group at every launch, so a
        loaded state dict's flag decides, as it does for ``torch.optim.Adam``."""
        return bool(self.hyper.get("decoupled_weight_decay", False))

    def _per_param_extra(self):
        return {"step": torch.tensor(float(self._steps))}

    def _dyn_values(self):
        h = self.hyper
        step = self._steps + 1
        lr = float(h["lr"])
        bc1 = 1.0 - float(h["betas"][0]) ** step
        bc2 = 1.0 - float(h["betas"][1]) ** step
        if self.decoupled:
            return (-(lr / bc1), bc2 ** 0.5, 1.0 - lr * float(h["weight_decay"]))
        return (-(lr / bc1), bc2 ** 0.5)

    def _launch(self, lo, hi, grad_scale, coef):
        h = self.hyper
        p, g, lp = self._slices(lo, hi)
        vmax = self._state("max_exp_avg_sq")[lo:hi] if h["amsgrad"] else None
        kernel = KERNELS.adamw if self.decoupled else KERNELS.adam
        kernel(p, g, self._state("exp_avg")[lo:hi], self._state("exp_avg_sq")[lo:hi], vmax,
               lp, hi - lo, lr=float(h["lr"]), beta1=float(h["betas"][0]),
               beta2=float(h["betas"][1]), eps=float(h["eps"]),
               wd=float(h["weight_decay"]), step=self._steps + 1,
               grad_scale=grad_scale, grad_scale_dev=coef, dyn=self._dyn)

    def _launch_mt(self, table, grad_scale):
        h = self.hyper
        kernel = KERNELS.adamw_mt if self.decoupled else KERNELS.adam_mt
        kernel(self.arena.master, self._state("exp_avg"), self._state("exp_avg_sq"),
               self._state("max_exp_avg_sq") if h["amsgrad"] else None, self.arena.lp, table,
               lr=float(h["lr"]), beta1=float(h["betas"][0]), beta2=float(h["betas"][1]),
               eps=float(h["eps"]), wd=float(h["weight_decay"]), step=self._steps + 1,
               grad_scale=grad_scale, dyn=self._dyn)

    def _launch_nvls(self, lo, hi, grad_scale):
        h = self.hyper
        mc_g, mc_out = self._nvls_ptrs(lo)
        vmax = self._state("max_exp_avg_sq")[lo:hi] if h["amsgrad"] else None
        kernel = KERNELS.nvls_adamw if self.decoupled else KERNELS.nvls_adam
        kernel(self.arena.master[lo:hi], self._state("exp_avg")[lo:hi],
               self._state("exp_avg_sq")[lo:hi], vmax, mc_g, mc_out, hi - lo, self.nvls,
               lr=float(h["lr"]), beta1=float(h["betas"][0]), beta2=float(h["betas"][1]),
               eps=float(h["eps"]), wd=float(h["weight_decay"]), step=self._steps + 1,
               grad_scale=grad_scale, g_dtype=KERNELS.dtype_code(self.arena.grad.dtype),
               dyn=self._dyn)


class FusedAdamW(FusedAdam):
    """``torch.optim.AdamW``: Adam with decoupled weight decay (p *= 1 - lr*wd, the gradient is
    not decayed).  As in torch, a thin subclass whose flag stays True whatever a loaded state
    dict says.  The default ``weight_decay`` here is the caller's (``OptimOpts.weightDecay``
    through ``create_fused_optimizer``); torch's own default of 1e-2 is not substituted."""

    def __init__(self, arena, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False):
        super().__init__(arena, lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad,
                         decoupled_weight_decay=True)

    def load_state_dict(self, state_dict: Dict[str, Any]) -> None:
        super().load_state_dict(state_dict)
        self.hyper["decoupled_weight_decay"] = True


class FusedRMSprop(FusedArenaOptimizer):
    STATE_NAMES = (("square_avg", "square_avg"), ("momentum_buffer", "momentum_buffer"))

    def __init__(self, arena, lr, alpha=0.99, eps=1e-8, weight_decay=0.0, momentum=0.0):
        super().__init__(arena, dict(lr=lr, momentum=momentum, alpha=alpha, eps=eps,
                                     centered=False, weight_decay=weight_decay, capturable=False,
                                     foreach=None, maximize=False, differentiable=False))

    def _per_param_extra(self):
        return {"step": torch.tensor(float(self._steps))}

    def _launch(self, lo, hi, grad_scale, coef):
        h = self.hyper
        p, g, lp = self._slices(lo, hi)
        mu = float(h["momentum"])
        buf = self._state("momentum_buffer")[lo:hi] if mu != 0.0 else None
        KERNELS.rmsprop(p, g, self._state("square_avg")[lo:hi], buf, lp, hi - lo,
                        lr=float(h["lr"]), alpha=float(h["alpha"]), eps=float(h["eps"]),
                        wd=float(h["weight_decay"]), mu=mu, grad_scale=grad_scale,
                        grad_scale_dev=coef, dyn=self._dyn)

    def _launch_mt(self, table, grad_scale):
        h = self.hyper
        mu = float(h["momentum"])
        KERNELS.rmsprop_mt(self.arena.master, self._state("square_avg"),
                           self._state("momentum_buffer") if mu != 0.0 else None, self.arena.lp, table,
                           lr=float(h["lr"]), alpha=float(h["alpha"]), eps=float(h["eps"]),
                           wd=float(h["weight_decay"]), mu=mu, grad_scale=grad_scale, dyn=self._dyn)

    def _launch_nvls(self, lo, hi, grad_scale):
        h = self.hyper
        mu = float(h["momentum"])
        mc_g, mc_out = self._nvls_ptrs(lo)
        buf = self._state("momentum_buffer")[lo:hi] if mu != 0.0 else None
        KERNELS.nvls_rmsprop(self.arena.master[lo:hi], self._state("square_avg")[lo:hi], buf, mc_g,
                             mc_out, hi - lo, self.nvls, lr=float(h["lr"]), alpha=float(h["alpha"]),
                             eps=float(h["eps"]), wd=float(h["weight_decay"]), mu=mu,
                             grad_scale=grad_scale,
                             g_dtype=KERNELS.dtype_code(self.arena.grad.dtype), dyn=self._dyn)


def check_decoupled_weight_decay(optim_opts: OptimOpts, decoupled_weight_decay: bool) -> None:
    """Decoupled weight decay exists for Adam only (torch 2.11 has no such flag for SGD/RMSprop)."""
    if decoupled_weight_decay and optim_opts.algo != OptAlgorithm.ADAM:
        raise ValueError("decoupled_weight_decay=True needs OptimOpts.algo == OptAlgorithm.ADAM "
                         "(AdamW); got %s" % getattr(optim_opts.algo, "value", optim_opts.algo))


def create_fused_optimizer(arena: ParamArena, optim_opts: OptimOpts, *,
                           decoupled_weight_decay: bool = False) -> FusedArenaOptimizer:
    """Same dispatch and argument mapping as the reference's ``_create_optimizer``.
    ``decoupled_weight_decay=True`` with ``OptAlgorithm.ADAM`` gives AdamW, with
    ``OptimOpts.weightDecay`` as the decoupled coefficient; with any other algorithm it is a
    ``ValueError``."""
    check_decoupled_weight_decay(optim_opts, decoupled_weight_decay)
    algo = optim_opts.algo
    if algo == OptAlgorithm.RMSPROP:
        return FusedRMSprop(arena, lr=optim_opts.lr, momentum=optim_opts.momentum,
                            weight_decay=optim_opts.weightDecay)
    if algo == OptAlgorithm.SGD:
        return FusedSGD(arena, lr=optim_opts.lr, momentum=optim_opts.momentum,
                        weight_decay=optim_opts.weightDecay)
    if algo == OptAlgorithm.ADAM:
        cls = FusedAdamW if decoupled_weight_decay else FusedAdam
        return cls(arena, lr=optim_opts.lr, weight_decay=optim_opts.weightDecay,
                   eps=optim_opts.epsilon, amsgrad=optim_opts.amsgrad)
    raise ValueError("Unknown optimization algorithm type")
