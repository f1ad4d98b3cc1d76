"""TEST INFRASTRUCTURE — what the UNMODIFIED reference returns for the API-parity scenarios of
``tests/test_oracle_pinning.py`` and ``tests/test_indexed_dataset.py``, recorded once so that the
tests compare this package against it without the reference being present:

    python -m oracle.reference_cases          # needs the reference (oracle/ref_shim.py)

Every scenario below takes the modules it exercises as arguments; ``main()`` runs it on the
reference's modules and writes ``tests/golden/reference_cases/<case>.pt`` (tensors, lists, dicts,
tuples and scalars only: read back with ``torch.load(..., weights_only=True)``), and the tests run
the same function on this package's modules and compare.  The checkpoint scenario stores the
reference's four checkpoint files themselves, next to the inputs they were written from.
"""
import io
import os
import random
import shutil
import sys
import tempfile
from typing import NamedTuple

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
OUT = os.path.join(REPO, "tests", "golden", "reference_cases")
CHECKPOINT_DIR = os.path.join(OUT, "checkpoint")
CHECKPOINT_FILES = [".checkpoint.pth", ".checkpoint.pth.annotate_param", ".checkpoint.pth.model",
                    ".checkpoint.pth.test_data"]
SAMPLER_STATE_CONFIGS = [("err_MSE", "DESC"), ("score", "ASC"), ("score", "DESC")]
CRITERION_KINDS = ["parallel", "uncertainty", "gradnorm", "masked"]
INDEXED_CASES = [("float32", (3, 4), 5), ("uint8", (2, 3, 5), 7), ("int64", (), 4), ("float64", (128,), 3),
                 ("int16", (1,), 1), ("int8", (4, 1, 2), 9), ("int32", (17,), 33)]


def load(name):
    return torch.load(os.path.join(OUT, name + ".pt"), weights_only=True)


def plain(obj):
    """numpy arrays / scalars -> tensors / Python scalars, recursively (what ``weights_only`` reads)."""
    if isinstance(obj, np.ndarray):
        return torch.from_numpy(np.array(obj, order="C"))
    if isinstance(obj, np.generic):
        return obj.item()
    if isinstance(obj, dict):
        return {k: plain(v) for k, v in obj.items()}
    if isinstance(obj, tuple):
        return tuple(plain(v) for v in obj)
    if isinstance(obj, list):
        return [plain(v) for v in obj]
    if torch.is_tensor(obj):
        return obj.detach().clone()
    return obj


# ---- SamplerState: retained minibatches -> per-sample metrics, random picks, worst-k ---------------

def sampler_state_record(state):
    """What a caller reads back from a folded SamplerState (the scenario of
    oracle/make_sampler_state_golden.py)."""
    def sample(s):
        return {"data": [a.clone() for a in s.data], "output": [a.clone() for a in s.output],
                "target": [a[0].clone() for a in s.target], "metric": {k: float(v) for k, v in s.metric.items()}}
    return {"n_samples": int(state.n_samples),
            "data_metric": {k: plain(np.asarray(v)) for k, v in state.data_metric.items()},
            "random_ids": [int(s.meta["index"]) for s in state.random_samples],
            "worst_ids": [int(s.meta["index"]) for s in state.worst_samples],
            "samples": {int(s.meta["index"]): sample(s) for s in state.worst_samples + state.random_samples}}


def reference_sampler_state(metric_name, ordering):
    from oracle import make_sampler_state_golden as gen
    import frldistml.scaffold.solver_worker as ref_sw
    from frldistml.scaffold.problem import Ordering
    batches, total = gen.scenario()

    class FakeLoader:
        sampler = list(range(total))

    random.seed(gen.PY_SEED)
    state = ref_sw.SamplerState(gen.make_problem(Ordering, metric_name, ordering), FakeLoader,
                                list(range(total)), torch.device("cpu"), gen.N_VIS)
    gen.drive(state, batches)
    return sampler_state_record(state)


# ---- the criterion classes' own composition --------------------------------------------------------

def criterion_trace(kind, c, m, t):
    """Four SGD steps of a 2-task model through the criterion class ``kind`` of module ``c``:
    per step the total loss, the sub-losses and every parameter's gradient; then the parameters."""
    torch.manual_seed(3)
    trunk = torch.nn.Sequential(m.ListSelect(sel_index=0, num_elements=1), torch.nn.Linear(6, 8),
                                torch.nn.ReLU(), torch.nn.Linear(8, 8), torch.nn.ReLU())
    model = m.MultiTaskModel(trunk, [torch.nn.Linear(8, 3), torch.nn.Linear(8, 5)])
    mods = [torch.nn.MSELoss(), torch.nn.CrossEntropyLoss()]
    names, weights = ["reg", "cls"], [0.5, 2.0]
    if kind == "parallel":
        crit = c.ParallelCriterion(mods, weights, names)
    elif kind == "uncertainty":
        crit = c.UncertaintyWeightedCriterion(mods, [t.LossType.MSE, t.LossType.CrossEntropy], names, weights)
    elif kind == "gradnorm":
        crit = c.GradNormWeightedCriterion(mods, names, alpha=1.5, base_weights=weights)
    else:
        crit = c.ParallelCriterion([c.MaskedLoss(torch.nn.MSELoss()), torch.nn.CrossEntropyLoss()], weights, names)

    g = torch.Generator().manual_seed(4)
    steps = []
    for k in range(4):
        x = torch.randn(12, 6, generator=g)
        y_reg, y_cls = torch.randn(12, 3, generator=g), torch.randint(0, 5, (12,), generator=g)
        mask = (torch.rand(12, 3, generator=g) > 0.4) if k != 2 else torch.zeros(12, 3, dtype=torch.bool)
        steps.append((x, y_reg, y_cls, mask))

    params = list(model.parameters()) + list(crit.parameters())
    opt = torch.optim.SGD(params, lr=0.05, momentum=0.9)
    trace = []
    for x, y_reg, y_cls, mask in steps:
        out = model([x])
        if kind == "gradnorm":
            crit.set_shared_params(model.final_shared_params(out))
        tgt = [(y_reg, mask) if kind == "masked" else (y_reg,), (y_cls,)]
        total, sub = crit(out, tgt)
        opt.zero_grad()
        total.backward()
        trace.append((total.detach().clone(), {k: v.detach().clone() for k, v in sub.items()},
                      [p.grad.detach().clone() for p in params]))
        opt.step()
    return {"steps": trace, "params": [p.detach().clone() for p in params]}


# ---- parent-side aggregation of the per-rank epoch summaries ---------------------------------------

AGGREGATION_PER_RANK = [   # (nSamples, losses, metrics) per split, three ranks with unequal sample counts
    {"training": (100, {"reg": 0.5, "cls": 2.25}, {"reg_MSE": 0.04, "cls_err": 0.25, "pose_MSE_deg": 9.0}),
     "testing": (10, {"reg": 0.7, "cls": 2.0}, {"reg_MSE": 0.09, "cls_err": 0.5, "pose_MSE_deg": -1.0})},
    {"training": (60, {"reg": 0.25, "cls": 1.75}, {"reg_MSE": 0.01, "cls_err": 0.125, "pose_MSE_deg": 4.0}),
     "testing": (30, {"reg": 0.1, "cls": 3.0}, {"reg_MSE": 0.16, "cls_err": 0.75, "pose_MSE_deg": -1.0})},
    {"training": (7, {"reg": 1.5, "cls": 0.5}, {"reg_MSE": 0.25, "cls_err": 1.0, "pose_MSE_deg": 1.0}),
     "testing": (3, {"reg": 0.3, "cls": 1.0}, {"reg_MSE": 0.0, "cls_err": 0.0, "pose_MSE_deg": -1.0})},
]


def aggregate_ranks(solver_mod, sw_mod, t):
    class DS:
        def __init__(self, split):
            self.data_type = split

    class P:
        datasets = [DS(t.Split.TRAIN), DS(t.Split.TEST)]

    fracs = []
    for rank in AGGREGATION_PER_RANK:
        perf = {t.Split(name): sw_mod.FractionalEpochSplitPerformanceSummary(
                    nSamples=n, losses=dict(losses), metrics=dict(metrics), samples=[],
                    worstSamples=[], testIO=[])
                for name, (n, losses, metrics) in rank.items()}
        fracs.append(sw_mod.FractionalPerformanceSummary(
            epoch=3, modelBuffer=b"", optimizerStateBuffer=b"", performance=perf))
    ro = t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm.SGD), batchSize=4)
    out = solver_mod.Solver._aggregate_fractional_results(ro, P(), fracs)
    return {split.value: (dict(s.losses), dict(s.metrics)) for split, s in out.items()}


# ---- checkpoint files written by the parent --------------------------------------------------------

class CheckpointAnno(NamedTuple):
    scale: float = 2.0
    names: tuple = ("a", "b")


class CheckpointProblem:
    anno_param = CheckpointAnno()


def checkpoint_inputs():
    """(model bytes, optimizer-state bytes, test samples) handed to ``Solver._save_checkpoint``."""
    torch.manual_seed(1)
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.BatchNorm1d(5), torch.nn.ReLU(),
                                torch.nn.Linear(5, 3))
    opt = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-5)
    for _ in range(3):
        opt.zero_grad()
        model(torch.randn(8, 6)).square().mean().backward()
        opt.step()
    model.eval()
    buf = io.BytesIO()
    torch.save(model, buf)
    model_bytes = buf.getvalue()
    buf = io.BytesIO()
    torch.save(opt.state_dict(), buf)
    optim_bytes = buf.getvalue()
    samples = [dict(data=[torch.randn(6)], target=[(torch.randn(3),)], meta={"index": torch.tensor(i)},
                    output=[torch.randn(3)], metric={"m": 0.5}) for i in range(2)]
    return model_bytes, optim_bytes, samples


def stored_checkpoint_inputs():
    """The inputs the stored reference checkpoint was written from."""
    with open(os.path.join(CHECKPOINT_DIR, "input.model"), "rb") as f:
        model_bytes = f.read()
    with open(os.path.join(CHECKPOINT_DIR, "input.optimizer"), "rb") as f:
        optim_bytes = f.read()
    samples = torch.load(os.path.join(CHECKPOINT_DIR, "input.samples"), weights_only=True)
    return model_bytes, optim_bytes, samples


def write_checkpoint(solver_mod, sw_mod, t, save_dir, inputs):
    model_bytes, optim_bytes, samples = inputs
    io_samples = [sw_mod.SingleSample(**s) for s in samples]
    perf = {t.Split.TRAIN: sw_mod.FractionalEpochSplitPerformanceSummary(
                nSamples=10, losses={}, metrics={}, samples=[], worstSamples=[], testIO=[]),
            t.Split.TEST: sw_mod.FractionalEpochSplitPerformanceSummary(
                nSamples=4, losses={}, metrics={}, samples=[], worstSamples=[], testIO=io_samples)}
    frac = sw_mod.FractionalPerformanceSummary(epoch=7, modelBuffer=model_bytes,
                                               optimizerStateBuffer=optim_bytes, performance=perf)
    ro = t.RunOpts(optim=t.OptimOpts(algo=t.OptAlgorithm.SGD), batchSize=4)
    solver_mod.Solver._save_checkpoint(7, save_dir, ro, CheckpointProblem(), [frac], ".checkpoint.pth")


# ---- initialModelPath: strict and partial loads ----------------------------------------------------

def init_net(width):
    torch.manual_seed(width)
    return torch.nn.Sequential(torch.nn.Linear(4, width), torch.nn.ReLU(), torch.nn.Linear(width, 2))


def write_initial_model(path):
    """A checkpoint with one unexpected key and one legacy serialised Parameter."""
    state = dict(init_net(5).state_dict())
    state["extra.weight"] = torch.ones(3)
    state["0.weight"] = torch.nn.Parameter(state["0.weight"].clone())
    torch.save({"state_dict": state}, path)


def initial_model_loads(load_model_state, path, read_stdout):
    """Partial loads into a same-width and a different-width net (weights and the warnings
    printed), then whether the strict load refuses the unexpected key."""
    target, other = init_net(5), init_net(7)
    read_stdout()
    load_model_state(target, path, strict=False)
    load_model_state(other, path, strict=False)
    lines = [l for l in read_stdout().splitlines() if l.startswith("Warning")]
    try:
        load_model_state(init_net(5), path, strict=True)
        strict_raises = False
    except RuntimeError:
        strict_raises = True
    read_stdout()
    return {"target": dict(target.state_dict()), "other": dict(other.state_dict()), "warnings": lines,
            "strict_raises": strict_raises}


# ---- the synthetic MultiTaskProblem built against an API namespace --------------------------------

def multitask_problem_plumbing(pkg):
    """Per-sample items, model structure and initial weights, criterion composition, merged metric
    hooks and rankable metric of the toy Problem instantiated against package ``pkg``."""
    import frl_b200  # noqa: F401
    from frl_b200 import synthetic
    ns = synthetic.api_namespace(pkg)
    problem = synthetic.make_toy_problem(ns, "/tmp/unused")
    torch.manual_seed(21)
    model = problem.get_model()
    crit = problem.get_criterion()
    items = [problem.datasets[0][i] for i in (0, 5, 511)] + [problem.datasets[1][3]]
    g = torch.Generator().manual_seed(2)
    out = [torch.randn(6, 4, generator=g), torch.randn(6, 10, generator=g)]
    tgt = [(torch.randn(6, 4, generator=g),), (torch.randint(0, 10, (6,), generator=g),)]
    meta = problem.refine_batch_meta({"index": torch.arange(6)})
    metrics = problem.compute_batch_metrics(meta=meta, target=tgt, output=out, device=torch.device("cpu"))
    with torch.no_grad():
        y = model([torch.ones(2, 64)])
    return plain(dict(
        model_type=type(model).__name__, crit_type=type(crit).__name__,
        state={k: v.clone() for k, v in model.state_dict().items()},
        names=list(crit.loss_names), weights=[float(w) for w in crit.loss_weights],
        loss_mods=[type(m).__name__ for m in crit.loss_modules],
        items=[(list(d), [tuple(x) for x in tg], {k: torch.as_tensor(v) for k, v in mt.items()})
               for d, tg, mt in items],
        metrics={k: np.asarray(v) for k, v in metrics.items()},
        rank=(problem.get_rankable_metric()[0], problem.get_rankable_metric()[1].name),
        epoch=problem.summarize_epoch_metrics({k: np.asarray(v) for k, v in metrics.items()}),
        meta_fields=tuple(meta._fields), y=[t.clone() for t in y],
        splits=[d.data_type.value for d in problem.datasets], lens=[len(d) for d in problem.datasets]))


# ---- indexed datasets: writer bytes and reader frames ----------------------------------------------

def indexed_frames():
    rs = np.random.RandomState(7)
    return [(dt, shape, [np.asarray(rs.randn(*shape) * 50).astype(dt) for _ in range(n)])
            for dt, shape, n in INDEXED_CASES]


def write_indexed(writer_cls, frames):
    idx, binf = io.BytesIO(), io.BytesIO()
    w = writer_cls(idxfile=idx, binfile=binf)
    for f in frames:
        w.push_back(f)
    w.flush()
    return idx.getvalue(), binf.getvalue()


def write_concat_parts(folder):
    """Three two-field indexed datasets of 5, 1 and 7 samples under ``folder/part<k>``."""
    import frl_b200  # noqa: F401
    from frl_b200 import indexed_dataset as idm
    rs = np.random.RandomState(9)
    for k, n in enumerate([5, 1, 7]):
        idm.write_fields(os.path.join(folder, "part%d" % k),
                         {"a": rs.randn(n, 3).astype(np.float32), "b": rs.randint(0, 9, (n, 2)).astype(np.int64)})


class AccessRecorder:
    def __init__(self, log, offset=0, field=None):
        self.log, self.offset, self.field = log, offset, field

    def with_dataset_global_offset(self, offset):
        return AccessRecorder(self.log, offset, self.field)

    def with_multifield_dataset_field(self, field):
        self.log.append((self.offset, field))
        return AccessRecorder(self.log, self.offset, field)


CONCAT_PICKS = [12, 0, 5, 5, 3]


def concat_and_subset(concat, subset_cls):
    """Raw and transformed items of a Concat dataset, the accessor calls it forwards to its parts,
    and the items of a Subset over it."""
    rec = {"len": len(concat), "raw": [dict(concat.get_raw_item(i)) for i in range(len(concat))],
           "items": [dict(concat[i]) for i in range(len(concat))], "accessor_log": []}
    concat.set_accessor(AccessRecorder(rec["accessor_log"]))
    sub = subset_cls(concat, CONCAT_PICKS)
    rec["subset_len"] = len(sub)
    rec["subset"] = [dict(sub[j]) for j in range(len(sub))]
    return plain(rec)


# ---- recording -------------------------------------------------------------------------------------

def main():
    import contextlib
    from oracle.ref_shim import import_reference
    import_reference()
    import frldistml.scaffold.criteria as ref_c
    import frldistml.scaffold.model as ref_m
    import frldistml.scaffold.solver as ref_solver
    import frldistml.scaffold.solver_worker as ref_sw
    import frldistml.scaffold.types as ref_t
    import frldistml.scaffold.storage_layers.dataset as ref_ds
    from frldistml.scaffold.indexed_dataset import MultifieldIndexedDataset as RefMulti
    from frldistml.scaffold.storage import StoragePath
    from frldistml.scaffold.storage_layers.dataset import IndexedDatasetWriter as RefWriter
    from frldistml.scaffold.storage_layers.posix_storage import PosixIndexedDatasetReader as RefReader

    os.makedirs(CHECKPOINT_DIR, exist_ok=True)

    def save(name, obj):
        torch.save(obj, os.path.join(OUT, name + ".pt"))

    for metric_name, ordering in SAMPLER_STATE_CONFIGS:
        save("sampler_state_%s_%s" % (metric_name, ordering), reference_sampler_state(metric_name, ordering))
    for kind in CRITERION_KINDS:
        save("criterion_%s" % kind, criterion_trace(kind, ref_c, ref_m, ref_t))
    save("rank_aggregation", aggregate_ranks(ref_solver, ref_sw, ref_t))

    tmp = tempfile.mkdtemp(prefix="frl_reference_cases_")
    try:
        model_bytes, optim_bytes, samples = inputs = checkpoint_inputs()
        for name, blob in (("input.model", model_bytes), ("input.optimizer", optim_bytes)):
            with open(os.path.join(CHECKPOINT_DIR, name), "wb") as f:
                f.write(blob)
        torch.save(samples, os.path.join(CHECKPOINT_DIR, "input.samples"))
        write_checkpoint(ref_solver, ref_sw, ref_t, StoragePath(tmp), inputs)
        assert sorted(os.listdir(tmp)) == CHECKPOINT_FILES
        for name in CHECKPOINT_FILES:
            shutil.copyfile(os.path.join(tmp, name), os.path.join(CHECKPOINT_DIR, name))

        path = os.path.join(tmp, "init.pth")
        write_initial_model(path)
        buf = io.StringIO()

        def read_stdout():
            text = buf.getvalue()
            buf.seek(0)
            buf.truncate()
            return text
        with contextlib.redirect_stdout(buf):
            rec = initial_model_loads(ref_solver._load_model_state, path, read_stdout)
        save("initial_model_loading", rec)

        cases = []
        for dt, shape, frames in indexed_frames():
            idx, binf = write_indexed(RefWriter, frames)
            ip, bp = os.path.join(tmp, "x.idx"), os.path.join(tmp, "x.bin")
            with open(ip, "wb") as f:
                f.write(idx)
            with open(bp, "wb") as f:
                f.write(binf)
            r = RefReader(idxfile=StoragePath(ip), binfile=StoragePath(bp))
            cases.append({"idx": torch.tensor(list(idx), dtype=torch.uint8),
                          "bin": torch.tensor(list(binf), dtype=torch.uint8),
                          "len": len(r), "framesize": int(r.framesize), "dtype": str(r.dtype),
                          "frames": [plain(r[i]) for i in range(len(r))]})
        save("indexed_writer_reader", cases)

        write_concat_parts(tmp)
        parts = [RefMulti(StoragePath(os.path.join(tmp, "part%d" % k)), fields=["a", "b"], filenames=["a", "b"])
                 for k in range(3)]
        save("concat_subset", concat_and_subset(ref_ds.ConcatMultifieldDataset(parts), ref_ds.SubsetMultifieldDataset))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    save("multitask_problem", multitask_problem_plumbing("frldistml.scaffold"))
    print("wrote", OUT, sorted(os.listdir(OUT)))


if __name__ == "__main__":
    main()
