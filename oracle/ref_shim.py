"""TEST INFRASTRUCTURE ONLY -- never imported by the product path (biscuit_b200/).

Import shim that loads the UNMODIFIED reference package `biscuit` from a checkout of the
original project named by the environment variable BISCUIT_REFERENCE_ROOT, so its
`threshold.apply / detect / from_cv` can be executed as the ground truth for the
thresholding half of the hot path (SURVEY.md App. C).

The reference imports matplotlib / seaborn / skmisc / slideflow at module import time
(reference biscuit/__init__.py:1-2, threshold.py:2-10, utils.py:6-9); none of those is
installed here and none is on the arithmetic path, so they are stubbed in
``sys.modules``.  sklearn / pandas / numpy / scipy are the REAL installed packages.

The reference is not part of this repository: only the `oracle/make_golden*.py` scripts
(output committed under tests/golden/) and the CPU-side live-reference tests (skipped
unless BISCUIT_REFERENCE_ROOT is set) may call :func:`load_reference`.
"""
import importlib
import logging
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("BISCUIT_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "biscuit", "threshold.py"))


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules[name] = mod
    return mod


def load_reference():
    """Returns the reference `biscuit` package (imported once, cached)."""
    if "biscuit" in sys.modules and getattr(sys.modules["biscuit"], "_is_reference", False):
        return sys.modules["biscuit"]
    if not reference_available():
        raise RuntimeError(f"reference not found: set BISCUIT_REFERENCE_ROOT to a checkout of the original biscuit "
                           f"project (now {REFERENCE_ROOT!r})")

    log = logging.getLogger("slideflow_stub")
    log.addHandler(logging.NullHandler())
    log.propagate = False
    if not hasattr(log, "warn"):
        log.warn = log.warning

    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors", "matplotlib.ticker",
                 "seaborn", "skmisc"):
        if name not in sys.modules:
            m = _stub(name)
            m.__path__ = []
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].colors = sys.modules["matplotlib.colors"]
    sys.modules["matplotlib"].ticker = sys.modules["matplotlib.ticker"]
    sys.modules["matplotlib.ticker"].__dict__.setdefault("PercentFormatter", object)
    if "skmisc.loess" not in sys.modules:
        _stub("skmisc.loess", loess=object)

    class _ModelParams:  # reference biscuit/hp.py:3 only needs a kwargs-accepting class
        def __init__(self, **kw):
            self.__dict__.update(kw)

    if "slideflow" not in sys.modules:
        def _manifest_slides(model_path, dataset=None):
            # documented behaviour of sf.util.get_slides_from_model_manifest: slide_manifest.csv in the model
            # folder or its parent, optional dataset filter (only the row COUNT reaches the reference's output)
            import csv
            for folder in (model_path, os.path.dirname(os.path.normpath(model_path))):
                path = os.path.join(folder, "slide_manifest.csv")
                if os.path.exists(path):
                    with open(path, newline="") as f:
                        return [r["slide"] for r in csv.DictReader(f) if dataset is None or r["dataset"] == dataset]
            raise OSError(f"no slide manifest for {model_path}")

        sf_util = _stub("slideflow.util", log=log, path_to_ext=lambda p: p.rsplit(".", 1)[-1],
                        bold=lambda t: t, get_slides_from_model_manifest=_manifest_slides)
        sf_model = _stub("slideflow.model", ModelParams=_ModelParams)
        sf = _stub("slideflow", util=sf_util, model=sf_model, Project=type("Project", (), {}))
        sf.__path__ = []

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    mod = importlib.import_module("biscuit")
    mod._is_reference = True
    importlib.import_module("biscuit.threshold")
    return mod
