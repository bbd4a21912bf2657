"""ORACLE side — test / benchmark infrastructure, NOT product code.

Stages and imports the UNMODIFIED reference (tqch/ddpm-torch @ b60eb8d) so that the parity fixtures, the reference arm of
``bench.py`` (``--impl reference``, ``cpu_baseline.kind = "reference"``) and the stock torch-CUDA comparison run the
reference's own code rather than the restatement in ``oracle/ddpm_ref.py``.

* ``stage()``  — build-container only: copies ``/root/reference/{ddpm_torch/, ddim.py, configs/}`` byte for byte into the
  git-ignored ``oracle/_ref/`` (listed in .gitignore, NOT in .gpurunignore, so it travels to the GPU box like a built
  ``.so``; it never enters the history).  The reference is pure Python with no ``setup.py`` / ``pyproject.toml``
  (SURVEY.md §1), so "installing" it is this copy.  Called by ``__graft_entry__.build()``.
* ``load()``   — imports it from ``oracle/_ref`` (only ``stage()`` reads the upstream checkout) with the one stub the
  image needs: ``ddpm_torch/utils/__init__.py:1-2`` imports matplotlib, which is not
  installed (SURVEY.md §8c).  Nothing of the reference is modified.

Only tests/, __graft_entry__, bench.py's reference legs and oracle/gen_golden.py may import this module.
"""
import os
import shutil
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
STAGED = os.path.join(HERE, "_ref")
UPSTREAM = "/root/reference"
_ITEMS = ("ddpm_torch", "ddim.py", "configs")


def stage(src=UPSTREAM, dst=STAGED):
    """Copy the reference's importable files into oracle/_ref (idempotent).  Returns the path, or None if src is absent.
    Contents only, not modes: the upstream files are read-only, and a copy that kept that could not be refreshed or
    removed by its owner."""
    if not os.path.isdir(os.path.join(src, "ddpm_torch")):
        return dst if available() else None
    os.makedirs(dst, exist_ok=True)
    for it in _ITEMS:
        s, d = os.path.join(src, it), os.path.join(dst, it)
        if os.path.isdir(s):
            for dirpath, dirnames, filenames in os.walk(s):
                dirnames[:] = [n for n in dirnames if n != "__pycache__"]
                out = os.path.join(d, os.path.relpath(dirpath, s))
                os.makedirs(out, exist_ok=True)
                for f in filenames:
                    if not f.endswith(".pyc"):
                        shutil.copyfile(os.path.join(dirpath, f), os.path.join(out, f))
        elif os.path.exists(s):
            shutil.copyfile(s, d)
    return dst


def available():
    return os.path.isdir(os.path.join(STAGED, "ddpm_torch"))


def root():
    return STAGED if available() else None


def load():
    """-> (ddpm_torch, ddim) modules of the unmodified reference.  Raises RuntimeError when it is not staged."""
    r = root()
    if r is None:
        raise RuntimeError("reference not staged: run `python -c 'import __graft_entry__ as g; g.build()'` in the build container")
    if "matplotlib" not in sys.modules:
        try:
            import matplotlib  # noqa: F401
        except ImportError:
            m = types.ModuleType("matplotlib"); m.rcParams = {}
            p = types.ModuleType("matplotlib.pyplot"); m.pyplot = p
            sys.modules["matplotlib"] = m; sys.modules["matplotlib.pyplot"] = p
    if r not in sys.path:
        sys.path.insert(0, r)
    import ddpm_torch
    import ddim
    return ddpm_torch, ddim


def config(name):
    """configs/<name>.json of the reference as a dict."""
    import json
    with open(os.path.join(root(), "configs", name + ".json")) as f:
        return json.load(f)
