"""Single-node convenience entry (reference local_solver.py:62-104): file:// rendezvous, a
fresh group name, run ``Solver.solve`` to the end and return the last epoch's summary.  The
reference's optional plotly notebook export is a visualisation add-on outside the hot path."""
import logging
import os
import pwd
import uuid
from typing import Optional

from .problem import Problem
from .solver import PerformanceSummary, Solver
from .types import Precision, RunOpts

logger = logging.getLogger(__name__)

SYNC_FILE = "/tmp/frl_dist_ml_sync" + "." + pwd.getpwuid(os.getuid()).pw_name


class LocalSolver:
    @classmethod
    def solve(cls, run_opts: RunOpts, problem: Problem, save_notebook: bool = False,
              precision: Optional[Precision] = None, graph: Optional[bool] = None,
              decoupled_weight_decay: bool = False) -> PerformanceSummary:
        if save_notebook:
            logger.warning("save_notebook is not supported by frl_b200 (visualisation only)")
        # a stale rendezvous file from a crashed run would poison the file:// store
        if os.path.exists(SYNC_FILE):
            os.remove(SYNC_FILE)
        open(SYNC_FILE, "w+").close()
        group_name = uuid.uuid4().hex
        logger.info("Group name: " + str(group_name))
        last: Optional[PerformanceSummary] = None
        for last in Solver.solve(run_opts, problem, group_name=group_name,
                                 init_method="file://" + SYNC_FILE, precision=precision,
                                 graph=graph, decoupled_weight_decay=decoupled_weight_decay):
            pass
        return last
