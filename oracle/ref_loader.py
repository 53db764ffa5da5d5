"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

Loads the *unmodified* reference modules on the CPU -- from the checkout HBR_REFERENCE_DIR names, else from the
verbatim copy __graft_entry__.build() stages in oracle/_ref (git-ignored) -- so that
(a) `oracle/make_golden.py` can generate the committed fixtures in tests/golden/ and
(b) bench.py's reference arm and the drop-in script tests run the reference itself (without a copy they use
    oracle/port.py or skip).

The shims are environmental only (SURVEY.md appendix B); no reference arithmetic is touched:
  * h5py / matplotlib are imported-but-unused by vol_renderer.py:4,6 and helper.py:7-8 -> empty stubs
  * numpy>=2 raises OverflowError for np.array([.., 2654435761, ..], dtype=np.int32)
    (hash_encoding.py:24); the pinned numpy 1.23 wraps to -1640531535 -> restore the wrap
  * MLP_3D.__init__ calls max_bound.to('cuda') (test_hash.py:25-26) -> duck-typed bound on CPU
"""
import contextlib
import io
import os
import sys
import types

import numpy as np

STAGED_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REF_DIR = os.environ.get("HBR_REFERENCE_DIR") or STAGED_DIR


def available() -> bool:
    return os.path.isfile(os.path.join(REF_DIR, "hash_encoding.py"))


class _NumpyInt32Wrap:
    """numpy facade whose array(..., dtype=int32) wraps like numpy 1.x did."""

    def __getattr__(self, k):
        return getattr(np, k)

    def array(self, obj, dtype=None, **kw):
        if dtype is np.int32:
            return np.array(obj, dtype=np.int64).astype(np.int32)
        return np.array(obj, dtype=dtype, **kw)


class Bound:
    """Stands in for the bbox tensors handed to MLP_3D on a CUDA-less host."""

    def __init__(self, t):
        self.t = t

    def to(self, *a, **k):
        return self.t


_cache = {}


def load():
    """Returns a namespace with the reference modules (hash_encoding, encoder, helper, test_hash, vol_renderer)."""
    if "ns" in _cache:
        return _cache["ns"]
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_DIR}")
    for n in ("h5py", "matplotlib", "matplotlib.pyplot", "matplotlib.lines"):
        if n not in sys.modules:
            sys.modules[n] = types.ModuleType(n)
    sys.modules["matplotlib.lines"].Line2D = object
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].lines = sys.modules["matplotlib.lines"]
    if "tmp_encoder" not in sys.modules:
        sys.modules["tmp_encoder"] = types.ModuleType("tmp_encoder")

    # The reference modules have generic names (encoder, helper, ...). Import them under the
    # reference directory only, then take them back out of sys.modules so they can never shadow
    # (or be shadowed by) the drop-in modules of the same names.
    names = ("hash_encoding", "encoder", "test_hash", "helper", "vol_renderer")
    saved = {n: sys.modules.pop(n) for n in names if n in sys.modules}
    sys.path.insert(0, REF_DIR)
    ns = types.SimpleNamespace()
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            import hash_encoding  # noqa
            hash_encoding.np = _NumpyInt32Wrap()
            import encoder  # noqa
            import test_hash  # noqa
            import helper  # noqa
            import vol_renderer  # noqa
        for n in names:
            setattr(ns, n, sys.modules[n])
    finally:
        sys.path.remove(REF_DIR)
        for n in names:
            sys.modules.pop(n, None)
        sys.modules.update(saved)
    ns.Bound = Bound
    _cache["ns"] = ns
    return ns


@contextlib.contextmanager
def quiet():
    """The reference prints on its hot path (hash_encoding.py:38, helper.py:42,50, test_hash.py:58)."""
    with contextlib.redirect_stdout(io.StringIO()):
        yield
