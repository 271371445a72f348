"""TEST INFRASTRUCTURE ONLY -- imports the UNMODIFIED reference modules (from /root/reference in the build
container, from the verbatim copy under baseline/_ref/ elsewhere).  Used by `oracle/make_golden.py`, by the CPU tests that
pin `oracle/block_oracle.py` against the real reference, and by the CPU arm of bench.py (`cpu_baseline.kind = "reference"`).  Recipe from SURVEY.md section 8(c): put the shim packages first on sys.path, chdir to
reference `src/` (config paths are relative, reference src/config.py:12-13), `import gnn`.
"""
import contextlib
import importlib
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIM = os.path.join(_HERE, "ref_shim")
# Where the unmodified reference may live: an explicit override (PFS_REFERENCE_ROOT), a checkout of the reference, or a
# verbatim copy of its src/gnn.py + src/config.py under baseline/_ref/ (git-ignored) -- SURVEY.md section 8c, BASELINE.md
# section 4.
VENDORED_ROOT = os.path.join(os.path.dirname(_HERE), "baseline", "_ref")


def _find_root():
    for root in (os.environ.get("PFS_REFERENCE_ROOT"), "/root/reference", VENDORED_ROOT):
        if root and os.path.isfile(os.path.join(root, "src", "gnn.py")):
            return root
    return "/root/reference"


REFERENCE_ROOT = _find_root()


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "src", "gnn.py"))


@contextlib.contextmanager
def _patched_path():
    src = os.path.join(REFERENCE_ROOT, "src")
    saved_path, saved_cwd = list(sys.path), os.getcwd()
    saved_mods = {k: sys.modules.get(k) for k in ("gnn", "config", "train", "torch_scatter",
                                                  "torch_geometric", "torch_geometric.data",
                                                  "matplotlib", "matplotlib.pyplot")}
    for k in saved_mods:
        sys.modules.pop(k, None)
    sys.path[:0] = [_SHIM, src]
    os.chdir(src)
    try:
        yield
    finally:
        os.chdir(saved_cwd)
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v


_cache = {}


def load_reference_gnn():
    """Return the reference `gnn` module object (classes Block, GNN, EdgeModel, ...)."""
    if "gnn" not in _cache:
        if not reference_available():
            raise RuntimeError("reference sources not present at %s" % REFERENCE_ROOT)
        with _patched_path():
            _cache["gnn"] = importlib.import_module("gnn")
            _cache["config"] = sys.modules["config"]
    return _cache["gnn"]


def load_reference_train():
    """Return the reference `train` module (for softfloor / loss_function)."""
    if "train" not in _cache:
        load_reference_gnn()
        with _patched_path():
            sys.modules["gnn"] = _cache["gnn"]
            sys.modules["config"] = _cache["config"]
            _cache["train"] = importlib.import_module("train")
    return _cache["train"]
