"""Import the UNMODIFIED reference (``$CTR_REFERENCE_ROOT/deepctr_torch``).

Used by ``make_golden.py`` (fixture generation) and by ``bench.py --impl reference``; the tests only read
the fixtures it produced.

The reference hard-imports ``tensorflow.python.keras.callbacks`` (reference
``deepctr_torch/callbacks.py:2-4``, ``models/basemodel.py:22-25``); tensorflow is not installed,
so four stub modules are registered in ``sys.modules`` that expose this repo's own Keras-style
callbacks.  Every stub carries a real ``ModuleSpec`` (``torch._dynamo`` calls
``importlib.util.find_spec("tensorflow")`` when the first optimizer is built).
"""
import importlib.machinery
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("CTR_REFERENCE_ROOT", "")


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "deepctr_torch"))


def _install_tf_stub():
    if "tensorflow" in sys.modules and not getattr(sys.modules["tensorflow"], "_ctr_stub", False):
        return
    repo = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    if repo not in sys.path:
        sys.path.insert(0, repo)
    from deepctr_torch_b200 import callbacks as cb

    names = ["tensorflow", "tensorflow.python", "tensorflow.python.keras",
             "tensorflow.python.keras.callbacks"]
    mods = {}
    for name in names:
        m = types.ModuleType(name)
        m.__spec__ = importlib.machinery.ModuleSpec(name, loader=None, is_package=True)
        m.__path__ = []
        m._ctr_stub = True
        mods[name] = m
        sys.modules[name] = m
    mods["tensorflow"].python = mods["tensorflow.python"]
    mods["tensorflow.python"].keras = mods["tensorflow.python.keras"]
    mods["tensorflow.python.keras"].callbacks = mods["tensorflow.python.keras.callbacks"]
    leaf = mods["tensorflow.python.keras.callbacks"]
    leaf.CallbackList = cb.CallbackList
    leaf.History = cb.History
    leaf.EarlyStopping = cb.EarlyStopping
    leaf.ModelCheckpoint = cb.ModelCheckpoint
    leaf.Callback = cb.Callback


def _offline_requests():
    """Stand-in for ``requests`` while the reference is imported: its ``__init__`` asks PyPI for a newer release
    in a thread (reference ``utils.py:19-44``); this ``get`` fails at once, so no connection is ever opened."""
    m = types.ModuleType("requests")

    def get(*args, **kwargs):
        raise ConnectionError("network access is disabled while the reference is loaded")
    m.get = get
    m.codes = types.SimpleNamespace(ok=200)
    return m


def load_reference():
    """Return the imported reference package ``deepctr_torch`` (unmodified sources)."""
    if not reference_available():
        raise RuntimeError("reference tree not found at %r (set CTR_REFERENCE_ROOT)" % REFERENCE_ROOT)
    _install_tf_stub()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    saved = sys.modules.get("requests")
    sys.modules["requests"] = _offline_requests()
    try:
        import deepctr_torch  # noqa: E402  (the reference; prints one "check the latest version" notice)
    finally:
        if saved is None:
            del sys.modules["requests"]
        else:
            sys.modules["requests"] = saved
    return deepctr_torch
