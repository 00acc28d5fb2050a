"""Import the UNMODIFIED reference from ``/root/reference`` (build container only).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Only ``oracle/make_golden.py``
(fixture generation) calls this: the tests, ``smoke()`` and ``bench.py`` compare with
the reference through the fixtures it wrote under ``tests/golden/``.
"""
import importlib
import os
import sys
import warnings

REFERENCE_ROOT = os.environ.get("VRR_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "vit.py"))


def load():
    """Return the reference modules ``(vit, positional_encoding, rope_utils)``."""
    if not available():
        raise FileNotFoundError(f"reference not mounted at {REFERENCE_ROOT}")
    from . import _timm_stub
    try:
        import timm  # noqa: F401  (a real timm wins if it is ever installed)
    except ImportError:
        _timm_stub.install()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    warnings.filterwarnings("ignore", category=FutureWarning)
    vit = importlib.import_module("models.vit")
    pe = importlib.import_module("models.positional_encoding")
    ru = importlib.import_module("models.rope_utils")
    if not os.path.abspath(vit.__file__).startswith(os.path.abspath(REFERENCE_ROOT)):
        raise ImportError("'models' resolved to something other than the reference")
    return vit, pe, ru
