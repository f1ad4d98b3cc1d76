"""AdamW (``decoupled_weight_decay=True``) on the B200 kernels: K2, K2-mt and the whole step.

There is no reference-recorded golden data for AdamW (the reference has no such optimizer): the
authority is stock ``torch.optim.AdamW``, on the CPU for the kernels and the toy Problem, and on
the same GPU for the 54.7M-parameter MLP.  Bounds are those of the matching Adam tests
(``test_gpu_kernels.py``, ``test_gpu_solver.py``, ``test_gpu_mlp_parity.py``)."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

import frl_b200  # noqa: F401
from frl_b200 import _native, synthetic
from frl_b200.solver import Solver, SolverWorkerArgs
from frl_b200.types import Device, Precision
from oracle import ref_loop
from oracle.make_golden import BATCH, SEED

from adamw_oracle import adamw_step, make_optimizer

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HP = dict(beta1=0.9, beta2=0.999, eps=1e-8)


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


# ---- K2 ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 4099, (1 << 18) + 3])
@pytest.mark.parametrize("ams", [False, True])
@pytest.mark.parametrize("gdt,lp", [(torch.float32, False), (torch.bfloat16, True)])
def test_adamw_matches_oracle_and_torch_adamw(n, ams, gdt, lp):
    rs = np.random.RandomState(n % 991)
    p0 = rs.randn(n).astype(np.float32)
    p, m, v = _dev(p0), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    vmax = torch.zeros(n, device=DEV) if ams else None
    p_lp = torch.zeros(n, dtype=torch.bfloat16, device=DEV) if lp else None
    rp, rm, rv = p0.copy(), np.zeros(n, np.float32), np.zeros(n, np.float32)
    rvm = np.zeros(n, np.float32) if ams else None
    wd = 0.05
    ref = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    topt = torch.optim.AdamW([ref], lr=1e-3, weight_decay=wd, eps=1e-8, amsgrad=ams, foreach=False)
    for step, lr in enumerate([1e-3, 4e-3, 5e-4, 2e-3], start=1):
        g = (rs.randn(n) * (0.1 if step == 3 else 1.0)).astype(np.float32)
        gd = _dev(g, gdt)
        g_seen = gd.float().cpu().numpy()
        _native.adamw(p, gd, m, v, vmax, p_lp, n, lr=lr, wd=wd, step=step, **HP)
        rp, rm, rv, rvm = adamw_step(rp, g_seen, rm, rv, rvm, lr=lr, wd=wd, step=step, **HP)
        topt.param_groups[0]["lr"] = lr
        ref.grad = torch.from_numpy(g_seen.copy())
        topt.step()
    np.testing.assert_allclose(p.cpu().numpy(), rp, rtol=3e-6, atol=2e-7)
    np.testing.assert_allclose(m.cpu().numpy(), rm, rtol=3e-6, atol=1e-7)
    np.testing.assert_allclose(v.cpu().numpy(), rv, rtol=3e-6, atol=1e-9)
    if ams:
        np.testing.assert_allclose(vmax.cpu().numpy(), rvm, rtol=3e-6, atol=1e-9)
    # torch.optim.AdamW itself (two 1-ulp scatters apart: the kernel's and the restatement's)
    np.testing.assert_allclose(p.cpu().numpy(), ref.detach().numpy(), rtol=1e-5, atol=1e-6)
    if lp:
        assert torch.equal(p_lp, p.to(torch.bfloat16))


def _mt_case(seed):
    from test_gpu_kernels import _mt_case as case
    return case(seed=seed)


def test_dyn_block_overrides_the_by_value_scalars():
    """Graph replays freeze by-value arguments: with ``dyn`` the kernel must take -lr/bc1, sqrt(bc2)
    AND keep = 1-lr*wd from device memory.  Wrong by-value lr/step + a right dyn == a right
    by-value launch, bit for bit, for K2 and K2-mt."""
    n = 70001
    rs = np.random.RandomState(2)
    p0, g0 = rs.randn(n).astype(np.float32), rs.randn(n).astype(np.float32)
    lr, wd, step = 3e-3, 0.1, 4
    bc1, bc2 = 1 - 0.9 ** step, 1 - 0.999 ** step
    dyn = torch.tensor([-(lr / bc1), bc2 ** 0.5, 1 - lr * wd, 0.0], dtype=torch.float32, device=DEV)
    m0 = np.abs(rs.randn(n)).astype(np.float32) * 0.1
    v0 = np.abs(rs.randn(n)).astype(np.float32) * 0.01

    def flat(use_dyn):
        p, m, v = _dev(p0), _dev(m0), _dev(v0)
        _native.adamw(p, _dev(g0), m, v, None, None, n, lr=0.5 if use_dyn else lr, wd=wd,
                      step=1 if use_dyn else step, dyn=dyn if use_dyn else None, **HP)
        return p, m, v

    for a, b in zip(flat(True), flat(False)):
        assert torch.equal(a, b)
    slots, grads, table, na = _mt_case(5)
    pa = np.random.RandomState(3).randn(na).astype(np.float32)

    def mt(use_dyn):
        p, m, v = _dev(pa), torch.zeros(na, device=DEV), torch.zeros(na, device=DEV)
        _native.adamw_mt(p, m, v, None, None, table, lr=0.5 if use_dyn else lr, wd=wd,
                         step=1 if use_dyn else step, dyn=dyn if use_dyn else None, **HP)
        return p, m, v

    for a, b in zip(mt(True), mt(False)):
        assert torch.equal(a, b)
    # and the decay really comes from dyn[2]: another keep gives other weights
    dyn2 = dyn.clone()
    dyn2[2] = 1.0
    p = _dev(p0)
    _native.adamw(p, _dev(g0), _dev(m0), _dev(v0), None, None, n, lr=lr, wd=wd, step=step, dyn=dyn2, **HP)
    assert not torch.equal(p, flat(False)[0])


@pytest.mark.parametrize("ams", [False, True])
@pytest.mark.parametrize("lp", [False, True])
def test_multi_tensor_adamw_equals_flatten_then_flat_update(ams, lp):
    slots, grads, table, n = _mt_case(3)
    rs = np.random.RandomState(9)
    p0 = rs.randn(n).astype(np.float32)
    used = np.zeros(n, bool)
    for s in slots:
        used[s.offset:s.offset + s.numel] = True
    p0[~used] = 0.0
    flat_g = torch.zeros(n, device=DEV)
    _native.flatten_grads(table, flat_g, scale=1.0)

    def run(mt):
        p = _dev(p0)
        s0, s1, s2 = (torch.zeros(n, device=DEV) for _ in range(3))
        p_lp = torch.zeros(n, dtype=torch.bfloat16, device=DEV) if lp else None
        for step in range(3):
            kw = dict(lr=1e-2 * (step + 1), wd=0.05, step=step + 1, grad_scale=0.5, **HP)
            if mt:
                _native.adamw_mt(p, s0, s1, s2 if ams else None, p_lp, table, **kw)
            else:
                _native.adamw(p, flat_g, s0, s1, s2 if ams else None, p_lp, n, **kw)
        torch.cuda.synchronize()
        return p, s0, s1, s2, p_lp

    a, b = run(True), run(False)
    for s in slots:
        sl = slice(s.offset, s.offset + s.numel)
        for x, y in zip(a, b):
            if x is not None:
                assert torch.equal(x[sl], y[sl]), s.index


def test_adamw_at_baseline_size_properties():
    """Full MLP arena (54.7M elements + criterion slot): size-independent properties."""
    n = 54_703_144 + 24
    lr, wd = 1e-3, 0.1
    p0 = torch.randn(n, device=DEV)
    g = torch.randn(n, device=DEV)
    # (1) zero gradient, fresh state: the weight is only decayed, p' == p * fp32(1 - lr*wd) exactly
    p, m, v = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    lp = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    _native.adamw(p, torch.zeros_like(g), m, v, None, lp, n, lr=lr, wd=wd, step=1, **HP)
    keep = torch.tensor(1 - lr * wd, dtype=torch.float32, device=DEV)
    assert torch.equal(p, p0 * keep) and torch.equal(lp, p.to(torch.bfloat16))
    # (2) wd = 0: AdamW is Adam, bit for bit
    pa, ma, va = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    pb, mb, vb = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    for step in (1, 2):
        _native.adamw(pa, g, ma, va, None, None, n, lr=lr, wd=0.0, step=step, **HP)
        _native.adam(pb, g, mb, vb, None, None, n, lr=lr, wd=0.0, step=step, **HP)
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb)
    # (3) the device clip coefficient scales the gradient, not the decay: coef 0.5 on g is the
    #     same launch as g * 0.5 with no coefficient (and differs from a decay scaled as well)
    coef = torch.tensor([0.5], device=DEV)
    p1, m1, v1 = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    p2, m2, v2 = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    _native.adamw(p1, g, m1, v1, None, None, n, lr=lr, wd=wd, step=1, grad_scale_dev=coef, **HP)
    _native.adamw(p2, g * 0.5, m2, v2, None, None, n, lr=lr, wd=wd, step=1, **HP)
    assert torch.equal(p1, p2) and torch.equal(m1, m2) and torch.equal(v1, v2)
    # closed form of step 1 (m/sqrt(v) = sign(g) up to eps) against torch ops on the device
    want = p0 * keep - lr * (m1 / (v1.sqrt() / (1 - 0.999) ** 0.5 + 1e-8)) / (1 - 0.9)
    torch.testing.assert_close(p1, want, rtol=1e-6, atol=1e-6)


# ---- the whole step through Solver.solve --------------------------------------------------------

WD = 0.05       # a decoupled coefficient whose effect is visible (1 - lr*wd != 1 in fp32)
CFGS = {        # (lr, scheduler, nEpochs, clip, amsgrad)
    "drop": (0.003, "drop", 2, 0.0, False),
    "multistep_clip": (0.003, "multistep", 3, 1.0, False),
    "amsgrad": (0.003, "drop", 2, 0.0, True),
}


def _run_opts(ns, cfg, **over):
    lr, sched, n_epochs, clip, amsgrad = cfg
    t = ns.types
    optim = t.OptimOpts(algo=t.OptAlgorithm.ADAM, lr=lr, weightDecay=WD,
                        lr_scheduler=t.LRSchedulerOpts(algo=t.LRSchedulerAlgorithm(sched)),
                        gradientClip=clip, amsgrad=amsgrad)
    kw = dict(optim=optim, batchSize=BATCH, nEpochs=n_epochs, numThreads=0, singleThreaded=True,
              numVisualizedSamples=4)
    kw.update(over)
    return t.RunOpts(**kw)


def _oracle(ns, cfg, batch=BATCH, monkeypatch=None):
    """ref_loop.train on the CPU with torch.optim.AdamW in place of its optimizer."""
    lr, sched, n_epochs, clip, amsgrad = cfg
    problem = synthetic.make_toy_problem(ns, "/tmp/unused")
    spec = ref_loop.RunSpec(optim=ref_loop.OptimSpec(algo="adam", lr=lr, scheduler=sched, weight_decay=WD,
                                                     gradient_clip=clip, amsgrad=amsgrad),
                            batch_size=batch, n_epochs=n_epochs)
    monkeypatch.setattr(ref_loop, "make_optimizer",
                        lambda params, o: make_optimizer(params, o, decoupled_weight_decay=True))
    torch.manual_seed(SEED)
    model, crit = problem.get_model(), problem.get_criterion()
    datasets = [(d.data_type.value, d) for d in problem.datasets]
    trace = ref_loop.train(model, list(crit.loss_modules), list(crit.loss_weights), list(crit.loss_names),
                           datasets, spec)
    monkeypatch.undo()
    rows = np.concatenate([trace.losses[k] for k in sorted(
        trace.losses, key=lambda ek: (ek[0], 0 if ek[1] == "training" else 1))])
    return trace, rows, problem


def _solve(ns, cfg, **over):
    save_dir = tempfile.mkdtemp(prefix="frl_b200_adamw_")
    problem = synthetic.make_toy_problem(ns, save_dir)
    captured = {}
    orig = Solver.build_worker.__func__

    def spy(cls, args):
        worker, sched, ckpt = orig(cls, args)
        captured["worker"] = worker
        return worker, sched, ckpt

    Solver.build_worker = classmethod(spy)
    try:
        torch.manual_seed(SEED)
        list(Solver.solve(_run_opts(ns, cfg, **over), problem, group_name=None,
                          init_method="file:///tmp/unused", precision=Precision.FP32,
                          decoupled_weight_decay=True))
    finally:
        Solver.build_worker = classmethod(orig)
    return captured["worker"], problem, save_dir


def _check_against_oracle(worker, problem, save_dir, trace, want_rows):
    rows = np.concatenate([r for _, _, r in worker.loss_history])
    assert rows.shape == want_rows.shape
    np.testing.assert_allclose(rows, want_rows, rtol=1e-5, atol=1e-6)
    served = sum((trace.indices[k] for k in sorted(trace.indices) if k[1] == "training"), [])
    assert problem.datasets[0].served == served
    final = torch.load(os.path.join(save_dir, "final_model.pth"), weights_only=False)
    for got, want in zip(final["state_dict"].values(), trace.params):
        np.testing.assert_allclose(got.numpy(), want, rtol=2e-4, atol=2e-6)
    opt_sd = final["optimizer"]
    assert opt_sd["param_groups"][0]["decoupled_weight_decay"] is True
    return final


@pytest.mark.parametrize("name", sorted(CFGS))
def test_solver_adamw_matches_torch_adamw_oracle(ns, name, monkeypatch):
    trace, want_rows, _ = _oracle(ns, CFGS[name], monkeypatch=monkeypatch)
    before = _native.launch_count()
    worker, problem, save_dir = _solve(ns, CFGS[name])
    assert _native.launch_count() > before
    assert worker.optimizer.decoupled
    final = _check_against_oracle(worker, problem, save_dir, trace, want_rows)
    # final_model.pth's optimizer state loads into stock torch.optim.AdamW
    model = problem.get_model()
    model.load_state_dict(final["state_dict"])
    opt = torch.optim.AdamW(model.parameters())
    opt.load_state_dict(final["optimizer"])
    assert opt.param_groups[0]["weight_decay"] == WD


def test_graph_replay_with_per_bucket_updates_reads_keep_from_dyn(ns, monkeypatch):
    """CUDA-graph replay with the per-bucket updates inside the captured graph (eager update path,
    no clip), a warm-up schedule that changes lr every epoch (a stale keep = 1 - lr*wd would show)
    and a ragged last batch (an eager step after the capture)."""
    cfg = (0.003, "multistep", 3, 0.0, False)
    batch = 48                                            # 512 = 10 x 48 + 32: ragged last batch
    trace, want_rows, _ = _oracle(ns, cfg, batch=batch, monkeypatch=monkeypatch)
    monkeypatch.setenv("FRL_B200_CUDA_GRAPH", "1")
    monkeypatch.setenv("FRL_B200_EAGER_UPDATE", "1")
    # host-side AdamW launches, tagged with whether a stream capture was open
    host_calls = []
    for name in ("adamw", "adamw_mt"):
        real = getattr(_native, name)

        def counted(*a, _real=real, **kw):
            host_calls.append(torch.cuda.is_current_stream_capturing())
            return _real(*a, **kw)
        monkeypatch.setattr(_native, name, counted)
    worker, problem, save_dir = _solve(ns, cfg, batchSize=batch)
    assert worker.pipeline.eager and worker.graphed is not None
    n_graphs = len(worker.graphed._graphs)
    assert n_graphs >= 1
    n_train_steps = sum(len(r) for e, s, r in worker.loss_history if s == ns.Split.TRAIN)
    assert n_train_steps == 3 * 11                        # per epoch 10 full batches + 1 ragged one
    # the per-bucket updates were captured into the graph (they are nodes of it, reading dyn) ...
    captured = host_calls.count(True)
    assert captured > 0
    # ... and the replayed steps launched nothing from the host: only the 2 eager steps before
    # each capture and the ragged steps did
    per_step = captured // n_graphs
    assert host_calls.count(False) < n_train_steps * per_step / 2
    assert worker.optimizer._dyn is not None and len(worker.optimizer._dyn_last) == 3
    _check_against_oracle(worker, problem, save_dir, trace, want_rows)


def test_resume_from_adamw_checkpoint_continues_like_torch_adamw(ns):
    cfg = (0.003, "drop", 6, 0.0, False)
    save_dir = tempfile.mkdtemp(prefix="frl_b200_adamw_resume_")
    problem = synthetic.make_toy_problem(ns, save_dir)
    torch.manual_seed(SEED)
    gen = Solver.solve(_run_opts(ns, cfg), problem, group_name=None, init_method="file:///tmp/unused",
                       decoupled_weight_decay=True)
    for summary in gen:
        if summary.epoch == 5:
            break
    gen.close()
    ckpt = torch.load(os.path.join(save_dir, ".checkpoint.pth"), weights_only=False)
    assert ckpt["epoch"] == 5 and ckpt["optimizer"]["param_groups"][0]["decoupled_weight_decay"] is True
    # stock AdamW from the checkpoint, one step on the CPU
    ref_problem = synthetic.make_toy_problem(ns, "/tmp/unused")
    ref_model, ref_crit = ref_problem.get_model(), ref_problem.get_criterion()
    ref_model.load_state_dict(ckpt["state_dict"])
    ref_opt = torch.optim.AdamW(list(ref_model.parameters()) + list(ref_crit.parameters()))
    ref_opt.load_state_dict(ckpt["optimizer"])
    assert ref_opt.param_groups[0]["weight_decay"] == WD
    # the fused optimizer resumed from the same checkpoint, one step on the same batch
    problem2 = synthetic.make_toy_problem(ns, save_dir)
    args = SolverWorkerArgs(run_opts=_run_opts(ns, cfg), problem=problem2, save_dir=save_dir,
                            run_device=Device.GPU, node_idx=0, node_count=1, rank=0, local_rank=0,
                            world_size=1, group_name=None, init_method="", decoupled_weight_decay=True)
    worker, _, loaded = Solver.build_worker(args)
    assert loaded is not None and worker.optimizer.decoupled and worker.optimizer._steps > 0
    ds = problem2.datasets[0]
    batch = torch.utils.data.default_collate([ds[i] for i in range(BATCH)])
    worker.model.train()
    worker._pass_one_minibatch(0, ns.Split.TRAIN, [t.cuda() for t in batch[0]],
                               [tuple(t.cuda() for t in head) for head in batch[1]])
    torch.cuda.synchronize()
    ref_model.train()
    ref_loop.reference_minibatch(
        ref_model, lambda o, t: ref_loop.parallel_criterion(list(ref_crit.loss_modules), list(ref_crit.loss_weights),
                                                            list(ref_crit.loss_names), o, t),
        ref_opt, list(ref_model.parameters()), 0.0, batch[0], batch[1])
    for s, p in zip(sorted((s for s in worker.arena.slots if s.is_model), key=lambda s: s.index),
                    ref_model.parameters()):
        np.testing.assert_allclose(worker.arena.master_view(s).cpu().numpy(), p.detach().numpy(),
                                   rtol=1e-5, atol=1e-7)


def test_mlp_config_bf16_one_step_matches_stock_adamw_on_the_gpu(monkeypatch):
    """The 54.7M-parameter MLP at batch 64 in bf16: one fused AdamW step against stock
    torch.optim.AdamW under bf16 autocast on the same GPU."""
    from test_gpu_mlp_parity import BATCH as MB, DEPTH, N_CLASSES, REG_DIM, WIDTH, _batches
    monkeypatch.setenv("FRL_B200_CUDA_GRAPH", "0")
    lr = 1e-3
    ns = synthetic.api_namespace("frl_b200")
    t = ns.types
    torch.manual_seed(0)
    problem = synthetic.make_mlp_problem(ns, tempfile.mkdtemp(prefix="frl_b200_mlp_"), n_train=8, width=WIDTH,
                                         n_classes=N_CLASSES, reg_dim=REG_DIM, depth=DEPTH)
    run_opts = t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm.ADAM, lr=lr, weightDecay=WD), batchSize=MB,
                         nEpochs=1, numThreads=0, singleThreaded=True, numVisualizedSamples=0)
    args = SolverWorkerArgs(run_opts=run_opts, problem=problem, save_dir=problem.save_dir,
                            run_device=Device.GPU, node_idx=0, node_count=1, rank=0, local_rank=0,
                            world_size=1, group_name=None, init_method="", precision=Precision.BF16,
                            decoupled_weight_decay=True)
    worker, _, _ = Solver.build_worker(args)
    assert worker.arena.n_trainable == 54_703_144 and worker.optimizer.decoupled
    worker.model.train()
    worker.criterion.train()
    x, y, r = _batches()[0]
    _, total, sub, _ = worker._pass_one_minibatch(0, t.Split.TRAIN, [x.cuda()], [(y.cuda(),), (r.cuda(),)])
    loss_b200 = float(total.detach())
    torch.cuda.synchronize()
    got = [worker.arena.master_view(s).cpu() for s in sorted(worker.arena.slots, key=lambda s: s.index)
           if s.is_model]

    torch.manual_seed(0)
    problem2 = synthetic.make_mlp_problem(ns, "/tmp/unused", n_train=8, width=WIDTH, n_classes=N_CLASSES,
                                          reg_dim=REG_DIM, depth=DEPTH)
    stock = problem2.get_model().cuda()
    before = [p.detach().cpu().clone() for p in stock.parameters()]
    opt = torch.optim.AdamW(stock.parameters(), lr=lr, weight_decay=WD)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = stock([x.cuda()])
    loss = torch.nn.functional.cross_entropy(out[0].float(), y.cuda()) + \
        torch.nn.functional.mse_loss(out[1].float(), r.cuda())
    loss.backward()
    opt.step()
    torch.cuda.synchronize()
    assert loss_b200 == pytest.approx(float(loss), rel=1e-2)
    keep = np.float32(1 - lr * WD)
    for a, b, p0 in zip(got, (p.detach().cpu() for p in stock.parameters()), before):
        # AdamW's first step: p*keep - lr*sign(g) (up to eps); the sign of a rounding-level bf16
        # gradient entry is device noise, so compare the typical entry, and the decay exactly
        # where the update is the same
        d = (a - b).abs().flatten()[: 1 << 24]
        assert float(d.median()) <= 1e-6, tuple(b.shape)
        upd_a, upd_b = a - p0 * keep, b - p0 * keep
        same = (upd_a.sign() == upd_b.sign()).float().mean()
        assert float(same) >= 0.95, tuple(b.shape)


def test_multi_gpu_adamw_matches_oracle(tmp_path):
    """>= 2 GPUs only: AdamW through NCCL + K2, K7 (NVLS) and NCCL + clip vs torch.optim.AdamW on
    the global batch."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "run_ddp_adamw_vs_oracle.py")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port",
                          "29543", script], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("DDP_ADAMW_PARITY_OK") == (3 if "NVLS_AVAILABLE True" in out.stdout else 2)
