"""The oracle (oracle/ref_loop.py, optim_np.py, criteria_np.py) against the committed golden
vectors recorded from the live reference and against torch's own ops; this package's classes
against what the reference's classes returned on the same inputs (oracle/reference_cases.py)."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import criteria_np, optim_np, ref_loop
from oracle import reference_cases as rc
from oracle.make_golden import BATCH, CONFIGS, SEED, run_oracle


def _golden_rows(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_ref_loop_reproduces_reference_run(golden_dir, name):
    g = _golden_rows(golden_dir, name)
    trace, problem = run_oracle(name, CONFIGS[name])
    rows = np.concatenate([trace.losses[k] for k in sorted(
        trace.losses, key=lambda ek: (ek[0], 0 if ek[1] == "training" else 1))])
    # bit-exact on the machine that made the fixture; other CPUs may pick different SIMD paths
    np.testing.assert_allclose(rows, g["rows"], rtol=2e-6, atol=1e-7)
    served = sum((trace.indices[k] for k in sorted(trace.indices) if k[1] == "training"), [])
    assert served == list(g["served_train"])            # sample order: exact
    n_param = len([k for k in g.files if k.startswith("param_") and k != "param_names"])
    for i in range(n_param):
        np.testing.assert_allclose(trace.params[i], g["param_%02d" % i], rtol=2e-5, atol=2e-7)
    lrs = [lr for lr, e in zip(g["lr"], g["epoch"])]
    for lr, epoch in zip(lrs, g["epoch"]):
        assert lr == pytest.approx(trace.lrs[epoch - 1], rel=1e-12)


def test_lr_closed_forms_match_reference_tables(golden_dir):
    table = json.load(open(os.path.join(golden_dir, "lr_schedules.json")))
    for key, lrs in table.items():
        if key.startswith("kat_"):
            continue
        sched, n = key.split("_n")
        got = [ref_loop.lr_at_epoch(0.1, e, int(n), sched) for e in range(1, int(n) + 1)]
        assert got == pytest.approx(lrs, rel=1e-12)
    # the reference's own known-answer test (tests/test_solver.py:17-34)
    assert table["kat_resume60_adam_lr0.01_n75"] == [pytest.approx(0.001)]
    assert ref_loop.lr_at_epoch(0.01, 61, 75, "drop") == pytest.approx(0.001)


def test_sampler_restatement_matches_reference_lists(golden_dir):
    table = json.load(open(os.path.join(golden_dir, "samplers.json")))
    assert table["randperm_n10_w4_nodes1_e1"] == [[5, 0, 7], [6, 8, 4], [1, 9, 5], [2, 3, 6]]
    for key, per_rank in table.items():
        m = re.fullmatch(r"(\w+)_n(\d+)_w(\d+)_nodes(\d+)_e(\d+)", key)
        kind = m.group(1)
        n, w, nodes, e = (int(m.group(i)) for i in (2, 3, 4, 5))
        for rank, expect in enumerate(per_rank):
            node_size = w // nodes
            got = ref_loop.rank_indices(n, e, rank, w, kind, node_idx=rank // node_size,
                                        node_count=nodes)
            assert got == expect, key


def test_ref_loop_equals_live_reference_bitwise(golden_dir):
    """tests/golden/toy_sgd.npz holds what the reference's own LocalSolver.solve recorded."""
    name = "toy_sgd"
    live = _golden_rows(golden_dir, name)
    trace, _ = run_oracle(name, CONFIGS[name])
    rows = np.concatenate([trace.losses[k] for k in sorted(
        trace.losses, key=lambda ek: (ek[0], 0 if ek[1] == "training" else 1))])
    assert np.array_equal(rows, live["rows"])
    assert np.array_equal(trace.params[0], live["param_00"])


# ---- numpy update rules vs torch.optim (what the reference actually calls) --------------------

def _torch_steps(opt_cls, kwargs, p0, grads):
    p = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = opt_cls([p], **kwargs)
    for g in grads:
        p.grad = torch.from_numpy(g.copy())
        opt.step()
    return p.detach().numpy()


def test_numpy_rules_match_torch_optim():
    rs = np.random.RandomState(3)
    p0 = rs.randn(257).astype(np.float32)
    grads = [rs.randn(257).astype(np.float32) for _ in range(5)]
    # SGD momentum
    want = _torch_steps(torch.optim.SGD, dict(lr=0.01, momentum=0.9, weight_decay=1e-5), p0, grads)
    p, buf = p0.copy(), np.zeros_like(p0)
    for i, g in enumerate(grads):
        p, buf = optim_np.sgd_step(p, g, buf, lr=0.01, mu=0.9, dampening=0.0, wd=1e-5,
                                   first_step=(i == 0))
    np.testing.assert_allclose(p, want, rtol=1e-6, atol=1e-7)
    # Adam (+amsgrad)
    for ams in (False, True):
        want = _torch_steps(torch.optim.Adam, dict(lr=1e-3, weight_decay=1e-5, eps=1e-8,
                                                   amsgrad=ams), p0, grads)
        p, m, v = p0.copy(), np.zeros_like(p0), np.zeros_like(p0)
        vmax = np.zeros_like(p0) if ams else None
        for i, g in enumerate(grads):
            p, m, v, vmax = optim_np.adam_step(p, g, m, v, vmax, lr=1e-3, beta1=0.9, beta2=0.999,
                                               eps=1e-8, wd=1e-5, step=i + 1)
        np.testing.assert_allclose(p, want, rtol=2e-6, atol=1e-7)
    # RMSprop with and without momentum
    for mu in (0.9, 0.0):
        want = _torch_steps(torch.optim.RMSprop, dict(lr=1e-3, momentum=mu, weight_decay=1e-5),
                            p0, grads)
        p, sq, buf = p0.copy(), np.zeros_like(p0), np.zeros_like(p0)
        for g in grads:
            p, sq, buf = optim_np.rmsprop_step(p, g, sq, buf, lr=1e-3, alpha=0.99, eps=1e-8,
                                               wd=1e-5, mu=mu)
        np.testing.assert_allclose(p, want, rtol=2e-6, atol=1e-7)


def test_numpy_criteria_match_torch_losses():
    rs = np.random.RandomState(5)
    out = rs.randn(33, 7).astype(np.float32)
    tgt = rs.randn(33, 7).astype(np.float32)
    lab = rs.randint(0, 7, size=33)
    lab[3] = -100
    to, tt, tl = (torch.tensor(out, requires_grad=True), torch.tensor(tgt), torch.tensor(lab))
    l = torch.nn.functional.mse_loss(to, tt)
    l.backward()
    loss, grad = criteria_np.mse(out, tgt)
    assert loss == pytest.approx(l.item(), rel=1e-6)
    np.testing.assert_allclose(grad, to.grad.numpy(), rtol=1e-5, atol=1e-8)
    to.grad = None
    l = torch.nn.functional.cross_entropy(to, tl)
    l.backward()
    loss, grad = criteria_np.cross_entropy(out, lab)
    assert loss == pytest.approx(l.item(), rel=1e-6)
    np.testing.assert_allclose(grad, to.grad.numpy(), rtol=1e-5, atol=1e-8)
    # masked variants against the reference's gather formulation
    mask = rs.rand(33) > 0.5
    ref = ref_loop.masked_loss(torch.nn.MSELoss(), torch.tensor(out), torch.tensor(tgt),
                               torch.tensor(mask))
    assert criteria_np.mse(out, tgt, mask)[0] == pytest.approx(ref.item(), rel=1e-6)
    empty = np.zeros(33, dtype=bool)
    ref0 = ref_loop.masked_loss(torch.nn.CrossEntropyLoss(), torch.tensor(out), torch.tensor(lab).clamp(min=0),
                                torch.tensor(empty))
    assert criteria_np.cross_entropy(out, lab, empty)[0] == pytest.approx(ref0.item(), rel=1e-6)
    assert criteria_np.mse(out, tgt, empty)[0] == 0.0


def test_bf16_round_matches_torch():
    x = np.random.RandomState(1).randn(4097).astype(np.float32) * 3
    want = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(optim_np.bf16_round(x), want)


# ------------------------------------------------------------------------------------------------
# SURVEY §8 a16 — SamplerState (retained minibatches -> per-sample metrics, random picks, worst-k)
# against what the reference class returned on identical inputs (oracle/reference_cases.py)
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("metric_name,ordering", rc.SAMPLER_STATE_CONFIGS)
def test_sampler_state_matches_live_reference(metric_name, ordering):
    import random
    from oracle import make_sampler_state_golden as gen
    import frl_b200  # noqa: F401
    import frl_b200.solver_worker as my_sw
    from frl_b200.problem import Ordering as MyOrdering

    ref = rc.load("sampler_state_%s_%s" % (metric_name, ordering))
    batches, total = gen.scenario()
    random.seed(gen.PY_SEED)
    state = my_sw.SamplerState(gen.make_problem(MyOrdering, metric_name, ordering), total, total,
                               torch.device("cpu"), gen.N_VIS)
    gen.drive(state, batches)
    state.finish()
    mine = rc.sampler_state_record(state)

    assert mine["n_samples"] == ref["n_samples"] == total
    for k in ("err_MSE", "score"):
        np.testing.assert_array_equal(mine["data_metric"][k].numpy(), ref["data_metric"][k].numpy())
    assert mine["random_ids"] == ref["random_ids"] and len(ref["random_ids"]) == 6
    assert sorted(mine["worst_ids"]) == sorted(ref["worst_ids"])
    assert len(ref["worst_ids"]) == 6
    for i, s in mine["samples"].items():
        r = ref["samples"][i]
        for key in ("data", "output", "target"):
            assert len(s[key]) == len(r[key]) and all(torch.equal(a, b) for a, b in zip(s[key], r[key])), key
        assert s["metric"] == r["metric"]


# ------------------------------------------------------------------------------------------------
# SURVEY §8 a8-a11 — the criterion classes' own composition (what runs for arbitrary user losses,
# and what the fused kernels are checked against on the GPU) against what the reference classes
# computed (oracle/reference_cases.py)
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", rc.CRITERION_KINDS)
def test_criterion_classes_match_live_reference(kind):
    import frl_b200  # noqa: F401
    import frl_b200.criteria as my_c
    import frl_b200.model as my_m
    import frl_b200.types as my_t

    ref = rc.load("criterion_%s" % kind)
    mine = rc.criterion_trace(kind, my_c, my_m, my_t)
    assert len(mine["steps"]) == len(ref["steps"]) == 4
    for (rt, rs, rg), (mt, ms, mg) in zip(ref["steps"], mine["steps"]):
        assert torch.equal(mt, rt)
        assert list(ms) == list(rs) and all(torch.equal(ms[k], rs[k]) for k in rs)
        assert len(mg) == len(rg) and all(torch.equal(a, b) for a, b in zip(mg, rg))
    assert len(mine["params"]) == len(ref["params"])
    assert all(torch.equal(a, b) for a, b in zip(mine["params"], ref["params"]))


# ------------------------------------------------------------------------------------------------
# parent-side aggregation of the per-rank epoch summaries (reference solver.py:457-526): sample-
# weighted means over ranks, MSE -> RMSE renaming, invalid (negative) metrics passed through
# ------------------------------------------------------------------------------------------------

def test_rank_aggregation_matches_live_reference():
    import frl_b200  # noqa: F401
    import frl_b200.solver as my_solver
    import frl_b200.solver_worker as my_sw
    import frl_b200.types as my_t

    want = rc.load("rank_aggregation")
    got = rc.aggregate_ranks(my_solver, my_sw, my_t)
    assert got == want
    assert set(want["training"][1]) == {"reg_RMSE", "cls_err", "pose_RMSE_deg"}
    assert want["testing"][1]["pose_RMSE_deg"] == -1.0          # invalid metric: not square-rooted


# ------------------------------------------------------------------------------------------------
# checkpoint files written by the parent (reference solver.py:565-651): same four files, same
# contents, and each side's loader reads the other's checkpoint
# ------------------------------------------------------------------------------------------------

def test_checkpoint_files_match_live_reference(tmp_path):
    import frl_b200  # noqa: F401
    import frl_b200.solver as my_solver
    import frl_b200.solver_worker as my_sw
    import frl_b200.types as my_t

    # the reference's files, written from these very inputs
    ref_dir, my_dir = rc.CHECKPOINT_DIR, tmp_path / "mine"
    my_dir.mkdir()
    rc.write_checkpoint(my_solver, my_sw, my_t, str(my_dir), rc.stored_checkpoint_inputs())
    names = sorted(os.listdir(my_dir))
    assert names == rc.CHECKPOINT_FILES == [".checkpoint.pth", ".checkpoint.pth.annotate_param",
                                            ".checkpoint.pth.model", ".checkpoint.pth.test_data"]

    def same(a, b):
        if torch.is_tensor(a):
            return torch.is_tensor(b) and a.dtype == b.dtype and torch.equal(a, b)
        if isinstance(a, dict):
            return isinstance(b, dict) and list(a) == list(b) and all(same(a[k], b[k]) for k in a)
        if isinstance(a, (list, tuple)):
            return type(a) is type(b) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
        return a == b

    for n in (".checkpoint.pth", ".checkpoint.pth.test_data", ".checkpoint.pth.annotate_param"):
        a = torch.load(os.path.join(ref_dir, n), weights_only=False)
        b = torch.load(os.path.join(my_dir, n), weights_only=False)
        assert same(a, b), n
    whole_ref = torch.load(os.path.join(ref_dir, ".checkpoint.pth.model"), weights_only=False)
    whole_mine = torch.load(os.path.join(my_dir, ".checkpoint.pth.model"), weights_only=False)
    assert same(dict(whole_ref.state_dict()), dict(whole_mine.state_dict()))
    # this package's loader reads the reference's file; the reference's loader returns the
    # "epoch", "state_dict" and "optimizer" entries of what torch.load reads, and those entries of
    # this package's file were found equal to the reference's above
    with open(os.path.join(ref_dir, ".checkpoint.pth"), "rb") as f:
        back = my_solver.Solver._load_checkpoint(f)
    with open(os.path.join(my_dir, ".checkpoint.pth"), "rb") as f:
        got = my_solver.Solver._load_checkpoint(f)
    ref_ckpt = torch.load(os.path.join(ref_dir, ".checkpoint.pth"), weights_only=False)
    assert got.epoch == back.epoch == ref_ckpt["epoch"] == 7
    assert same(dict(got.modelState), dict(back.modelState)) and same(got.optimizerState, back.optimizerState)
    assert same(dict(back.modelState), dict(ref_ckpt["state_dict"])) and same(back.optimizerState, ref_ckpt["optimizer"])
    torch.optim.SGD(whole_mine.parameters(), lr=0.1, momentum=0.9).load_state_dict(got.optimizerState)


def test_initial_model_loading_matches_live_reference(tmp_path, capsys):
    """``initialModelPath`` (reference solver.py:122-159): strict load, and the partial load that
    copies what matches in name and shape and reports the rest — same weights, same messages."""
    import frl_b200  # noqa: F401
    import frl_b200.solver as my_solver

    path = str(tmp_path / "init.pth")
    rc.write_initial_model(path)
    want = rc.load("initial_model_loading")
    got = rc.initial_model_loads(my_solver._load_model_state, path, lambda: capsys.readouterr().out)
    ra, rb, rl = want["target"], want["other"], want["warnings"]
    ma, mb, ml = got["target"], got["other"], got["warnings"]
    assert list(ma) == list(ra) and list(mb) == list(rb)
    assert all(torch.equal(ra[k], ma[k]) for k in ra) and all(torch.equal(rb[k], mb[k]) for k in rb)
    assert ml == rl and len(rl) >= 4
    assert got["strict_raises"] and want["strict_raises"]              # unexpected key "extra.weight"
    assert torch.equal(ma["0.weight"], rc.init_net(5).state_dict()["0.weight"])


def test_multitask_problem_plumbing_matches_live_reference():
    """The same synthetic MultiTaskProblem source instantiated against this package and against
    the reference (SURVEY §8b: Problem/MultiTaskProblem/MultiTaskTransform/Task/MultiTaskModel):
    per-sample items, model structure and initial weights, criterion composition, merged metric
    hooks and rankable metric must coincide."""
    ref = rc.load("multitask_problem")
    mine = rc.multitask_problem_plumbing("frl_b200")
    for k in ("model_type", "crit_type", "names", "weights", "loss_mods", "rank", "epoch", "meta_fields",
              "splits", "lens"):
        assert mine[k] == ref[k], k
    assert list(mine["state"]) == list(ref["state"])
    assert all(torch.equal(mine["state"][k], ref["state"][k]) for k in ref["state"])
    assert len(mine["y"]) == len(ref["y"]) and all(torch.equal(a, b) for a, b in zip(mine["y"], ref["y"]))
    assert list(mine["metrics"]) == list(ref["metrics"])
    assert all(np.array_equal(mine["metrics"][k], ref["metrics"][k]) for k in ref["metrics"])
    assert len(mine["items"]) == len(ref["items"]) == 4
    for a, b in zip(mine["items"], ref["items"]):
        assert len(a) == len(b) == 3
        assert len(a[0]) == len(b[0]) and all(torch.equal(x, y) for x, y in zip(a[0], b[0]))   # data list
        assert len(a[1]) == len(b[1]) and all(torch.equal(x[0], y[0]) for x, y in zip(a[1], b[1]))  # targets
        assert list(a[2]) == list(b[2]) and all(torch.equal(a[2][k], b[2][k]) for k in a[2])
