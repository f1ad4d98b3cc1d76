"""Import the UNMODIFIED reference as the package ``frldistml.scaffold``.

TEST INFRASTRUCTURE.  Source: ``/root/reference`` where it exists (the build container), else the
archive ``oracle/build_ref.py`` packed into the git-ignored ``oracle/_ref/reference.zip`` (which
travels to the GPU box); used by ``oracle/make_golden.py`` to generate the committed fixtures, by
``oracle/reference_cases.py`` to record the reference's API-parity results, and by the
CPU arm of ``bench.py``.

What the shim does (SURVEY §8c), without touching the reference tree:
  * a temp dir with ``frldistml/__init__.py`` and a symlink ``frldistml/scaffold -> /root/reference``
    (the reference uses relative imports and its tests use that package name);
  * ``sys.modules`` stubs for two absent visualisation deps: ``plotly.graph_objs`` (types.py:20)
    and ``nbformat`` (local_solver.py:16);
  * ``TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD=1`` for the whole-module ``torch.load`` at solver.py:604.
"""
import os
import sys
import tempfile
import types

REFERENCE_DIR = "/root/reference"
REFERENCE_ZIP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "reference.zip")
_state = {}


def _tree_available() -> bool:
    return os.path.isdir(REFERENCE_DIR) and os.path.exists(os.path.join(REFERENCE_DIR, "solver.py"))


def reference_available() -> bool:
    return _tree_available() or os.path.exists(REFERENCE_ZIP)


def _stub_module(name: str, **attrs) -> types.ModuleType:
    mod = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(mod, k, v)
    sys.modules[name] = mod
    return mod


def import_reference():
    """Returns the imported ``frldistml.scaffold`` package (cached)."""
    if "pkg" in _state:
        return _state["pkg"]
    if not reference_available():
        raise RuntimeError("the reference is neither at /root/reference nor installed in oracle/_ref")
    os.environ["TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD"] = "1"

    if "plotly" not in sys.modules:
        class Figure(dict):
            pass
        plotly = _stub_module("plotly")
        plotly.graph_objs = _stub_module("plotly.graph_objs", Figure=Figure)
    if "nbformat" not in sys.modules:
        nb = _stub_module("nbformat", write=lambda *a, **k: None)
        nb.notebooknode = _stub_module("nbformat.notebooknode", NotebookNode=dict)
        nb.v4 = _stub_module("nbformat.v4", new_markdown_cell=lambda s: {"md": s},
                             new_code_cell=lambda s: {"code": s},
                             new_notebook=lambda cells=None: {"cells": cells})
    if "mock" not in sys.modules:
        import unittest.mock
        sys.modules["mock"] = unittest.mock

    # an frl_b200.install_reference_alias() made earlier in this process must not shadow the
    # real reference
    for k in [k for k in sys.modules if k == "frldistml" or k.startswith("frldistml.")]:
        del sys.modules[k]
    if _tree_available():
        root = tempfile.mkdtemp(prefix="frl_ref_shim_")
        os.makedirs(os.path.join(root, "frldistml"))
        open(os.path.join(root, "frldistml", "__init__.py"), "w").close()
        os.symlink(REFERENCE_DIR, os.path.join(root, "frldistml", "scaffold"))
        sys.path.insert(0, root)
        sys.dont_write_bytecode = True         # /root/reference is read-only
    else:
        sys.path.insert(0, REFERENCE_ZIP)      # zipimport: frldistml/scaffold/*.py inside
    import importlib
    pkg = importlib.import_module("frldistml.scaffold")
    for name in ("types", "criteria", "model", "lr_scheduler", "sampler", "transform", "task",
                 "problem", "multitask_problem", "solver_worker", "solver", "local_solver"):
        importlib.import_module("frldistml.scaffold." + name)
    _state["pkg"] = pkg
    return pkg
