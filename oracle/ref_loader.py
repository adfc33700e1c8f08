"""Load the reference's own Python modules from a checkout of it (``BCAD_REFERENCE_ROOT``) -- TEST INFRASTRUCTURE.

Used only by ``tests/golden/make_golden.py`` to generate the fixtures; the tests read those fixtures
and never need the reference itself.

The reference has import-time side effects that must not leak (SURVEY section 5):
``Classes/CNNModel.py:10`` opens a log file in cwd, ``:28`` replaces ``sys.stdout``,
``:587`` loads weights from a Windows path.  We exec the source truncated before that last
line, inside a temp cwd, and restore stdout.  ``explainability.py:11`` imports matplotlib
(unused, absent here) -> stubbed.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import tempfile
import types

REF_ROOT = os.environ.get("BCAD_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "Classes", "CNNModel.py"))


@contextlib.contextmanager
def _quiet_tmp_cwd():
    old_cwd, old_out = os.getcwd(), sys.stdout
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            yield
        finally:
            sys.stdout = old_out
            os.chdir(old_cwd)


def load_numpy_cnn() -> types.ModuleType:
    """Module namespace holding the reference ``CNNModel`` class and ``load_weights``."""
    path = os.path.join(REF_ROOT, "Classes", "CNNModel.py")
    src = open(path, encoding="utf-8").read()
    cut = src.index("Model = load_weights(")
    mod = types.ModuleType("ref_CNNModel")
    mod.__file__ = path
    with _quiet_tmp_cwd():
        exec(compile(src[:cut], path, "exec"), mod.__dict__)
        log = mod.__dict__.get("log_file")
        if log is not None:
            log.close()
    sys.stdout = sys.__stdout__ if isinstance(sys.stdout, mod.Logger) else sys.stdout
    return mod


def load_explainability() -> types.ModuleType:
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    path = os.path.join(REF_ROOT, "WebApplicationPrototype", "explainability.py")
    src = open(path, encoding="utf-8").read()
    mod = types.ModuleType("ref_explainability")
    mod.__file__ = path
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def load_adcnnm() -> types.ModuleType:
    path = os.path.join(REF_ROOT, "WebApplicationPrototype", "ADCNNM.py")
    src = open(path, encoding="utf-8").read()
    mod = types.ModuleType("ref_ADCNNM")
    mod.__file__ = path
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


@contextlib.contextmanager
def silenced():
    """The reference prints on construction / load; keep test output clean."""
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        yield buf
