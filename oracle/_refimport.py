"""TEST INFRASTRUCTURE ONLY — imports the *unmodified* reference modules from the directory named by RG_REFERENCE_DIR.

Only usable where a checkout of the original project is available; point RG_REFERENCE_DIR at it.  Used by
``oracle/gen_golden.py`` (fixture generation) and by ``tests/test_oracle_vs_reference.py`` (pins the
numpy restatements in ``oracle/`` against the real reference code).

The reference imports matplotlib (``lab3.py:20-22``, ``fun.py:5``), which is not installed here and is
never used on the hot path (plot helpers only), so empty stub modules are injected before import
(SURVEY.md section 8c).  ``sys.dont_write_bytecode`` keeps the read-only tree untouched.
"""
import contextlib
import importlib
import os
import sys
import types

REFERENCE_DIR = os.environ.get("RG_REFERENCE_DIR", "")


def reference_available() -> bool:
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "lab3.py"))


def _stub_matplotlib() -> None:
    if "matplotlib" in sys.modules:
        return
    try:
        import matplotlib  # noqa: F401  (real one present: nothing to do)
        return
    except Exception:
        pass
    names = ["matplotlib", "matplotlib.pyplot", "matplotlib.image", "matplotlib.patches",
             "mpl_toolkits", "mpl_toolkits.mplot3d"]
    for n in names:
        m = types.ModuleType(n)
        m.__path__ = []  # behave like a package so dotted imports resolve
        sys.modules[n] = m
    sys.modules["matplotlib.patches"].ConnectionPatch = object
    sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].image = sys.modules["matplotlib.image"]
    sys.modules["matplotlib"].patches = sys.modules["matplotlib.patches"]


@contextlib.contextmanager
def reference_cwd():
    """The reference opens its data with cwd-relative paths (``fun.py:85``, ``correspondences.py:12``)."""
    old = os.getcwd()
    os.chdir(REFERENCE_DIR)
    try:
        yield
    finally:
        os.chdir(old)


def import_reference(*names):
    """Import reference modules by flat name (``lab3``, ``fun``, ``ransac``, ``pnp`` ...)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_DIR}")
    _stub_matplotlib()
    sys.dont_write_bytecode = True
    added = False
    if REFERENCE_DIR not in sys.path:
        # appended (not prepended) so that the reference's flat names never shadow anything else;
        # callers that also use the drop-in flat modules must not mix both in one process.
        sys.path.append(REFERENCE_DIR)
        added = True
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mods = [importlib.import_module(n) for n in names]
    finally:
        if added:
            sys.path.remove(REFERENCE_DIR)
    return mods[0] if len(mods) == 1 else mods
