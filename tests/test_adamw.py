"""AdamW (``decoupled_weight_decay=True``) on the host side: the numpy restatement against
``torch.optim.AdamW``, the fused optimizer front and its torch-format checkpoints, the argument
validation of the entry points, and the two-rank bucket pipeline over gloo.  Kernel entry points
are the CPU test double (``adamw_oracle.AdamWKernelDouble``); the kernels themselves are checked
in ``test_gpu_adamw.py``."""
import inspect
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

import frl_b200  # noqa: F401
from frl_b200 import fused_optim, grad_sync, local_solver, solver
from frl_b200.arena import ParamArena
from frl_b200.types import OptAlgorithm, OptimOpts, RunOpts
from oracle.ref_loop import OptimSpec

from adamw_oracle import AdamWKernelDouble, adamw_step, make_optimizer


@pytest.fixture()
def double(monkeypatch):
    d = AdamWKernelDouble()
    monkeypatch.setattr(fused_optim, "KERNELS", d)
    monkeypatch.setattr(grad_sync, "KERNELS", d)
    return d


def _net(seed=0):
    torch.manual_seed(seed)
    return nn.Sequential(nn.Linear(7, 5), nn.ReLU(), nn.Linear(5, 3), nn.ReLU(), nn.Linear(3, 2))


# ---- the numpy restatement is torch.optim.AdamW ------------------------------------------------

@pytest.mark.parametrize("foreach", [False, True])
@pytest.mark.parametrize("amsgrad", [False, True])
def test_adamw_step_matches_torch_adamw(foreach, amsgrad):
    rng = np.random.default_rng(5)
    n = 4099
    p0 = rng.standard_normal(n).astype(np.float32)
    w = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    wd = 0.05
    opt = torch.optim.AdamW([w], lr=1e-3, weight_decay=wd, eps=1e-8, amsgrad=amsgrad, foreach=foreach)
    p, m, v = p0.copy(), np.zeros(n, np.float32), np.zeros(n, np.float32)
    vmax = np.zeros(n, np.float32) if amsgrad else None
    for step, lr in enumerate([1e-3, 3e-3, 2.5e-4, 7e-3, 1e-2, 5e-4], start=1):
        g = (rng.standard_normal(n) * (10.0 ** rng.uniform(-4, 1, n))).astype(np.float32)
        for grp in opt.param_groups:
            grp["lr"] = lr
        w.grad = torch.from_numpy(g.copy())
        opt.step()
        p, m, v, vmax = adamw_step(p, g, m, v, vmax, lr=lr, beta1=0.9, beta2=0.999, eps=1e-8, wd=wd,
                                   step=step)
        st = opt.state[w]
        np.testing.assert_allclose(p, w.detach().numpy(), rtol=2e-6, atol=1e-7)
        # the moments: 1-ulp scatter of lerp / addcmul, measured against the vector's scale (a
        # lerp that nearly cancels has a larger relative error than its operands)
        for mine, name in ((m, "exp_avg"), (v, "exp_avg_sq"), (vmax, "max_exp_avg_sq")):
            if mine is not None:
                want = st[name].numpy()
                np.testing.assert_allclose(mine, want, rtol=2e-6, atol=2e-6 * float(np.abs(want).max()))


def test_zero_decay_is_adam_and_decay_is_not_rescaled():
    """wd = 0: AdamW is Adam.  wd > 0: the decay of a weight with zero gradient and fresh state is
    exactly p * fp32(1 - lr*wd) (with coupled Adam it would be a whole step of size lr)."""
    from oracle.optim_np import adam_step
    rng = np.random.default_rng(1)
    p = rng.standard_normal(257).astype(np.float32)
    g = rng.standard_normal(257).astype(np.float32)
    z = np.zeros_like(p)
    kw = dict(lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, step=1)
    a = adam_step(p, g, z, z, None, wd=0.0, **kw)
    b = adamw_step(p, g, z, z, None, wd=0.0, **kw)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)
    out = adamw_step(p, z, z, z, None, wd=0.1, **kw)[0]
    assert np.array_equal(out, p * np.float32(1 - 1e-3 * 0.1))


# ---- fused optimizer front --------------------------------------------------------------------

def _train_both(net, ref, opt, ref_opt, steps, lrs=None):
    pipe = grad_sync.GradBucketPipeline(opt.arena, opt)
    x = torch.randn(16, 7, generator=torch.Generator().manual_seed(3))
    for step in range(steps):
        if lrs is not None:
            opt.param_groups[0]["lr"] = lrs[step]
            ref_opt.param_groups[0]["lr"] = lrs[step]
        pipe.begin_step()
        net(x).square().mean().backward()
        pipe.finish_step()
        ref_opt.zero_grad()
        ref(x).square().mean().backward()
        ref_opt.step()
    return pipe


@pytest.mark.parametrize("amsgrad", [False, True])
def test_fused_adamw_follows_torch_adamw_and_checkpoints_interchange(double, amsgrad):
    net, ref = _net(1), _net(1)
    opts = OptimOpts(algo=OptAlgorithm.ADAM, lr=0.01, weightDecay=0.02, amsgrad=amsgrad)
    arena = ParamArena(net.parameters(), device="cpu")
    opt = fused_optim.create_fused_optimizer(arena, opts, decoupled_weight_decay=True)
    assert isinstance(opt, fused_optim.FusedAdamW) and opt.decoupled
    ref_opt = make_optimizer(ref.parameters(), OptimSpec(algo="adam", lr=0.01, weight_decay=0.02,
                                                         amsgrad=amsgrad), decoupled_weight_decay=True)
    assert isinstance(ref_opt, torch.optim.AdamW)
    _train_both(net, ref, opt, ref_opt, 5, lrs=[0.01, 0.02, 0.005, 0.01, 0.001])
    assert {c[0] for c in double.calls} == {"adamw"}
    for a, b in zip(net.parameters(), ref.parameters()):
        np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-5, atol=1e-7)

    # state_dict: what torch.optim.AdamW emits — same group keys in the same order, same values
    sd, ref_sd = opt.state_dict(), ref_opt.state_dict()
    assert list(sd["param_groups"][0]) == list(ref_sd["param_groups"][0])
    assert sd["param_groups"][0] == ref_sd["param_groups"][0]
    assert sd["param_groups"][0]["decoupled_weight_decay"] is True
    assert list(sd["state"]) == list(ref_sd["state"])
    for k, entry in ref_sd["state"].items():
        assert list(sd["state"][k]) == list(entry)
        for name, val in entry.items():
            assert sd["state"][k][name].shape == val.shape and sd["state"][k][name].dtype == val.dtype
            if name == "step":
                assert float(sd["state"][k][name]) == float(val) == 5.0
            else:
                np.testing.assert_allclose(sd["state"][k][name].numpy(), val.numpy(), rtol=1e-4, atol=1e-9)

    # stock torch.optim.AdamW accepts it and keeps stepping in step with the fused optimizer
    net2 = _net(1)
    with torch.no_grad():
        for a, b in zip(net2.parameters(), net.parameters()):
            a.copy_(b)
    torch_opt = torch.optim.AdamW(net2.parameters())
    torch_opt.load_state_dict(sd)
    assert torch_opt.param_groups[0]["weight_decay"] == 0.02

    # round trip into a fresh FusedAdamW: identical vectors and step count
    net3 = _net(7)
    arena3 = ParamArena(net3.parameters(), device="cpu")
    opt3 = fused_optim.FusedAdamW(arena3, lr=0.5)
    opt3.load_state_dict(sd)
    assert opt3._steps == opt._steps == 5
    assert opt3.param_groups[0]["lr"] == opt.param_groups[0]["lr"]
    for name in opt._vec:
        assert torch.equal(opt3._vec[name], opt._vec[name]), name

    # one more step each: the resumed fused optimizer and torch.optim.AdamW agree
    with torch.no_grad():
        for a, b in zip(net3.parameters(), net.parameters()):
            a.copy_(b)
    pipe3 = grad_sync.GradBucketPipeline(arena3, opt3)
    x = torch.randn(16, 7, generator=torch.Generator().manual_seed(11))
    pipe3.begin_step(); net3(x).square().mean().backward(); pipe3.finish_step()
    torch_opt.zero_grad(); net2(x).square().mean().backward(); torch_opt.step()
    for a, b in zip(net3.parameters(), net2.parameters()):
        np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-5, atol=1e-7)


def test_coupled_adam_state_dict_still_loads_and_runs_coupled(double):
    ref = _net(2)
    opts = OptimOpts(algo=OptAlgorithm.ADAM, lr=0.01, weightDecay=0.02)
    ref_opt = torch.optim.Adam(ref.parameters(), lr=0.01, weight_decay=0.02)
    x = torch.randn(16, 7)
    for _ in range(2):
        ref_opt.zero_grad(); ref(x).square().mean().backward(); ref_opt.step()
    ref_sd = ref_opt.state_dict()
    ref_sd_nokey = {"state": ref_sd["state"],
                    "param_groups": [{k: v for k, v in ref_sd["param_groups"][0].items()
                                      if k != "decoupled_weight_decay"}]}
    for sd in (ref_sd, ref_sd_nokey):
        net = _net(2)
        with torch.no_grad():
            for a, b in zip(net.parameters(), ref.parameters()):
                a.copy_(b)
        arena = ParamArena(net.parameters(), device="cpu")
        opt = fused_optim.create_fused_optimizer(arena, opts)
        opt.load_state_dict(sd)
        assert not opt.decoupled and opt._steps == 2
        double.calls.clear()
        pipe = grad_sync.GradBucketPipeline(arena, opt)
        pipe.begin_step(); net(x).square().mean().backward(); pipe.finish_step()
        assert {c[0] for c in double.calls} == {"adam"}
    ref_opt.zero_grad(); ref(x).square().mean().backward(); ref_opt.step()
    for a, b in zip(net.parameters(), ref.parameters()):
        np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-5, atol=1e-7)


def test_loaded_flag_decides_like_torch(double):
    """torch.optim.Adam takes the loaded group's flag; torch.optim.AdamW stays decoupled."""
    net = _net(4)
    adamw_sd = torch.optim.AdamW(_net(4).parameters(), weight_decay=1e-3).state_dict()
    adam_sd = torch.optim.Adam(_net(4).parameters(), weight_decay=1e-3).state_dict()
    a = fused_optim.FusedAdam(ParamArena(net.parameters(), device="cpu"), lr=1e-3)
    a.load_state_dict(adamw_sd)
    assert a.decoupled
    b = fused_optim.FusedAdamW(ParamArena(_net(4).parameters(), device="cpu"), lr=1e-3)
    b.load_state_dict(adam_sd)
    assert b.decoupled and b.param_groups[0]["decoupled_weight_decay"] is True


def test_device_scalars_carry_one_minus_lr_wd():
    """Under CUDA-graph replay the kernels read lr-dependent scalars from the dyn block: AdamW's
    keep = 1 - lr*wd is slot 2 and follows the lr of the next step; coupled Adam leaves it 0."""
    arena = ParamArena(_net(0).parameters(), device="cpu")
    opt = fused_optim.FusedAdamW(arena, lr=1e-3, weight_decay=0.05)
    opt.enable_dynamic_scalars()
    assert opt._dyn[2].item() == np.float32(1 - 1e-3 * 0.05)
    opt.param_groups[0]["lr"] = 4e-3
    opt.begin_step()
    assert opt._dyn[2].item() == np.float32(1 - 4e-3 * 0.05)
    assert opt._dyn[0].item() == np.float32(-(4e-3 / (1 - 0.9)))
    coupled = fused_optim.FusedAdam(ParamArena(_net(0).parameters(), device="cpu"), lr=1e-3, weight_decay=0.05)
    coupled.enable_dynamic_scalars()
    assert coupled._dyn[2].item() == 0.0


# ---- argument validation ------------------------------------------------------------------------

@pytest.mark.parametrize("algo", [OptAlgorithm.SGD, OptAlgorithm.RMSPROP])
def test_flag_is_rejected_for_sgd_and_rmsprop(algo, monkeypatch):
    arena = ParamArena(_net(0).parameters(), device="cpu")
    with pytest.raises(ValueError, match="decoupled_weight_decay"):
        fused_optim.create_fused_optimizer(arena, OptimOpts(algo=algo), decoupled_weight_decay=True)
    # the entry point raises in the parent, before any device check or rank
    started = []
    monkeypatch.setattr(solver, "_cuda_device_count_without_poisoning_fork",
                        lambda: started.append("probe") or 1)
    run_opts = RunOpts(optim=OptimOpts(algo=algo), batchSize=8)
    with pytest.raises(ValueError, match="decoupled_weight_decay"):
        next(solver.Solver.solve(run_opts, problem=None, group_name=None, init_method="file:///tmp/x",
                                 decoupled_weight_decay=True))
    assert started == []


def test_flag_with_adam_passes_validation_and_defaults_change_nothing():
    run_opts = RunOpts(optim=OptimOpts(algo=OptAlgorithm.ADAM), batchSize=8, cpuonly=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        next(solver.Solver.solve(run_opts, problem=None, group_name=None, init_method="file:///tmp/x",
                                 decoupled_weight_decay=True))
    sig = inspect.signature(solver.Solver.solve)
    assert sig.parameters["decoupled_weight_decay"].kind == inspect.Parameter.KEYWORD_ONLY
    assert sig.parameters["decoupled_weight_decay"].default is False
    lsig = inspect.signature(local_solver.LocalSolver.solve)
    assert lsig.parameters["decoupled_weight_decay"].default is False
    assert solver.SolverWorkerArgs._fields[-1] == "decoupled_weight_decay"
    assert solver.SolverWorkerArgs._field_defaults["decoupled_weight_decay"] is False
    arena = ParamArena(_net(0).parameters(), device="cpu")
    opt = fused_optim.create_fused_optimizer(arena, OptimOpts(algo=OptAlgorithm.ADAM))
    assert type(opt) is fused_optim.FusedAdam and not opt.decoupled
    assert solver._update_rule_name(opt) == "Adam"
    assert solver._update_rule_name(fused_optim.FusedAdamW(arena, lr=1e-3, amsgrad=True)) == "AdamW (amsgrad)"


# ---- world_size 2 over gloo ---------------------------------------------------------------------

def _rank_main(rank, world, port, clip, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    d = AdamWKernelDouble()
    fused_optim.KERNELS = d
    grad_sync.KERNELS = d
    net = _net(10 + rank)                      # deliberately different: broadcast must fix it
    arena = ParamArena(net.parameters(), device="cpu")
    opt = fused_optim.create_fused_optimizer(arena, OptimOpts(algo=OptAlgorithm.ADAM, lr=0.05, weightDecay=0.1),
                                             decoupled_weight_decay=True)
    pipe = grad_sync.GradBucketPipeline(arena, opt, world_size=world, clip_norm=clip,
                                        bucket_cap_mb=0.0001, first_bucket_mb=0.00005)
    pipe.broadcast_parameters(src=0)
    assert len(pipe.buckets) > 1
    g = torch.Generator().manual_seed(99)
    for step in range(3):
        x = torch.randn(8 * world, 7, generator=g)
        pipe.begin_step()
        net(x[rank::world]).square().mean().backward()
        pipe.finish_step()
    assert {c[0] for c in d.calls} >= {"adamw"} and "adam" not in {c[0] for c in d.calls}
    torch.save([p.detach().clone() for p in net.parameters()], os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.parametrize("clip", [0.0, 0.01])
def test_two_rank_adamw_pipeline_equals_global_batch_training(tmp_path, clip):
    world = 2
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_rank_main, args=(world, port, clip, str(tmp_path)), nprocs=world, join=True)
    r0 = torch.load(tmp_path / "r0.pt")
    r1 = torch.load(tmp_path / "r1.pt")
    for a, b in zip(r0, r1):
        assert torch.equal(a, b)                               # replicas stay identical
    ref = _net(10)
    ref_opt = make_optimizer(ref.parameters(), OptimSpec(algo="adam", lr=0.05, weight_decay=0.1),
                             decoupled_weight_decay=True)
    g = torch.Generator().manual_seed(99)
    for step in range(3):
        x = torch.randn(8 * world, 7, generator=g)
        ref_opt.zero_grad()
        ref(x).square().mean().backward()
        if clip:
            torch.nn.utils.clip_grad_norm_(ref.parameters(), clip)
        ref_opt.step()
    for a, b in zip(r0, ref.parameters()):
        np.testing.assert_allclose(a.numpy(), b.detach().numpy(), rtol=2e-5, atol=1e-7)
