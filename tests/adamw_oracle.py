"""AdamW oracle for the tests: a numpy restatement of torch 2.11's decoupled-weight-decay Adam
step, a kernel test double that adds ``adamw`` to ``oracle.optim_np.KernelDouble``, and the
stock-PyTorch optimizer a run with ``decoupled_weight_decay=True`` is compared with.

The reference project has no AdamW, so there is no recorded golden data for it: the authority
is stock ``torch.optim.AdamW`` on the CPU, computed live by the tests (the same third-party
arithmetic ``oracle.ref_loop`` is pinned to for Adam, SGD and RMSprop).  The modules under
``oracle/`` stay the reference-pinned restatement they are."""
import numpy as np
import torch

from oracle.optim_np import KernelDouble, adam_step
from oracle.ref_loop import OptimSpec, make_optimizer as _ref_make_optimizer

f32 = np.float32


def adamw_step(p, g, m, v, vmax, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0):
    """torch/optim/adam.py _single_tensor_adam, ``decoupled_weight_decay`` branch:
    param.mul_(1 - lr * weight_decay) first (1 - lr*wd formed from Python floats, applied in
    fp32), then the Adam step of the decayed weight with the undecayed gradient."""
    p = (p.astype(f32) * f32(1 - lr * wd)).astype(f32)
    return adam_step(p, g, m, v, vmax, lr=lr, beta1=beta1, beta2=beta2, eps=eps, wd=0.0, step=step,
                     grad_scale=grad_scale)


class AdamWKernelDouble(KernelDouble):
    """``KernelDouble`` plus the AdamW entry point of ``frl_b200._native`` (CPU tensors)."""

    def adamw(self, p, g, m, v, vmax, p_lp, n, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0,
              grad_scale_dev=None, dyn=None):
        self.calls.append(("adamw", n))
        np_, nm, nv, nvm = adamw_step(self._np(p), self._np(g), self._np(m), self._np(v),
                                      self._np(vmax), lr=lr, beta1=beta1, beta2=beta2, eps=eps,
                                      wd=wd, step=step,
                                      grad_scale=self._scale(grad_scale, grad_scale_dev))
        self._store(p, np_); self._store(m, nm); self._store(v, nv); self._store(vmax, nvm)
        self._store(p_lp, np_)


def make_optimizer(params, o: OptimSpec, decoupled_weight_decay: bool = False) -> torch.optim.Optimizer:
    """``oracle.ref_loop.make_optimizer`` with torch's decoupled flag: ``algo="adam"`` and
    ``decoupled_weight_decay=True`` build ``torch.optim.AdamW`` with the spec's own weight decay
    (torch's AdamW default of 1e-2 is not substituted)."""
    if not decoupled_weight_decay:
        return _ref_make_optimizer(params, o)
    if o.algo != "adam":
        raise ValueError("decoupled weight decay exists for Adam only")
    return torch.optim.AdamW(params, lr=o.lr, weight_decay=o.weight_decay, eps=o.epsilon,
                             amsgrad=o.amsgrad)
