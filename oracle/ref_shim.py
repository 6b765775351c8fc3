"""Import shim that lets the UNMODIFIED reference (/root/reference) be imported in the build
container, where its optional third-party deps (rapidfuzz, matplotlib, seaborn) are absent.
TEST INFRASTRUCTURE -- used by tests/golden/make_golden.py, and by the GPU tests that run the reference's
orchestrator from the copy stage() makes (they skip where there is none)."""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("PFZ_REFERENCE_ROOT", "/root/reference")
# git-ignored copy of the reference's package, made by stage(): machines that only receive the working tree import it from here
STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "polyfuzz"))


def stage() -> bool:
    """Copy the reference's pure-Python package (REFERENCE_ROOT/polyfuzz) to STAGED_ROOT/polyfuzz.  Returns False and
    changes nothing when the reference is not readable here."""
    src = os.path.join(REFERENCE_ROOT, "polyfuzz")
    if not os.path.isdir(src) or os.path.abspath(REFERENCE_ROOT) == STAGED_ROOT:
        return False
    import shutil
    dst = os.path.join(STAGED_ROOT, "polyfuzz")
    shutil.rmtree(dst, ignore_errors=True)
    shutil.copytree(src, dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    return True


def install():
    """Register stub modules for the absent optional deps and put the reference on sys.path."""
    if not available():
        raise ImportError(f"reference not found at {REFERENCE_ROOT}")

    def _stub(name, **attrs):
        if name in sys.modules:
            return sys.modules[name]
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    def _absent(*_a, **_k):
        raise ModuleNotFoundError("stubbed third-party function (package not installed here)")

    try:
        import rapidfuzz  # noqa: F401
    except ModuleNotFoundError:
        fuzz = _stub("rapidfuzz.fuzz", ratio=_absent, WRatio=_absent)
        process = _stub("rapidfuzz.process", extractOne=_absent)
        _stub("rapidfuzz", fuzz=fuzz, process=process)
    try:
        import matplotlib  # noqa: F401
    except ModuleNotFoundError:
        plt = _stub("matplotlib.pyplot")
        gs = _stub("matplotlib.gridspec")
        cm = _stub("matplotlib.cm", get_cmap=_absent)
        lines = _stub("matplotlib.lines", Line2D=object)
        _stub("matplotlib", pyplot=plt, gridspec=gs, cm=cm, lines=lines)
    try:
        import seaborn  # noqa: F401
    except ModuleNotFoundError:
        _stub("seaborn")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
