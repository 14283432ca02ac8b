"""TEST INFRASTRUCTURE ONLY -- loads the *unmodified* reference classes from a checkout of the original
project (benoriol/hand_pose_sl) named by the environment variable B2H_REFERENCE_ROOT.

With that checkout available it is used to
 (a) validate the restatement in oracle/b2h_oracle.py (tests/test_oracle_vs_reference.py) and
 (b) generate the golden vectors committed under tests/golden/ (oracle/make_golden.py).
Without it the live comparisons skip; tests/test_oracle_golden.py checks the oracle against the stored
vectors.  Nothing in the product package imports this file.

Recipe (SURVEY.md §8c): the reference's package __init__ files import fairseq / h5py and two
classes that do not exist, so the three hot-path source files are loaded *by file path* with
empty stub modules registered for the absent third-party imports.  None of the stubs is
touched by the hot path.
"""
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("B2H_REFERENCE_ROOT", "")
_SRC = os.path.join(REF_ROOT, "body2hand", "src")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(_SRC, "models", "HandPoseModels.py"))


def _stub(name, **attrs):
    if name in sys.modules:
        mod = sys.modules[name]
    else:
        mod = types.ModuleType(name)
        mod.__b2h_stub__ = True
        sys.modules[name] = mod
    for k, v in attrs.items():
        if not hasattr(mod, k):
            setattr(mod, k, v)
    return mod


def _install_stubs():
    class _Dummy:  # never instantiated by the hot path
        def __init__(self, *a, **k):
            raise RuntimeError("fairseq stub: not part of the body2hand conv hot path")

    try:
        import fairseq  # noqa: F401  (absent in this image)
    except Exception:
        _stub("fairseq")
        _stub("fairseq.utils", get_available_activation_fns=lambda: ["relu"])
        sys.modules["fairseq"].utils = sys.modules["fairseq.utils"]
        _stub("fairseq.models")
        _stub("fairseq.models.fairseq_encoder", EncoderOut=_Dummy)
        _stub("fairseq.modules", FairseqDropout=_Dummy, LayerDropModuleList=_Dummy, LayerNorm=_Dummy,
              PositionalEmbedding=_Dummy, SinusoidalPositionalEmbedding=_Dummy,
              TransformerEncoderLayer=_Dummy)
    try:
        import h5py  # noqa: F401
    except Exception:
        _stub("h5py")


def _load(modname, relpath):
    path = os.path.join(_SRC, relpath)
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_cache = {}


def load():
    """Returns (models_mod, utils_mod, dataset_mod) = the reference's HandPoseModels.py,
    steps/utils.py and dataloaders/text_pose_dataset.py executed unmodified."""
    if not available():
        raise FileNotFoundError(f"no reference checkout: set B2H_REFERENCE_ROOT (now {REF_ROOT!r})")
    if not _cache:
        _install_stubs()
        _cache["models"] = _load("b2h_ref_HandPoseModels", "models/HandPoseModels.py")
        _cache["utils"] = _load("b2h_ref_steps_utils", "steps/utils.py")
        _cache["data"] = _load("b2h_ref_text_pose_dataset", "dataloaders/text_pose_dataset.py")
    return _cache["models"], _cache["utils"], _cache["data"]


def load_function(rel_path, name):
    """One top-level function of a reference file that cannot be imported as a module (steps/traintest.py uses
    package-relative imports and h5py): its source is taken UNMODIFIED from the file and executed with numpy / torch
    in scope.  TEST INFRASTRUCTURE ONLY."""
    import ast
    import numpy as np
    import torch
    if not available():
        raise FileNotFoundError(f"no reference checkout: set B2H_REFERENCE_ROOT (now {REF_ROOT!r})")
    path = os.path.join(REF_ROOT, "body2hand", "src", rel_path)
    src = open(path).read()
    for node in ast.parse(src).body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            ns = {"np": np, "torch": torch}
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
            return ns[name]
    raise KeyError(f"{name} not found in {path}")
