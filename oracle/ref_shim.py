"""ORACLE (test infrastructure only): import shim that loads the UNMODIFIED reference PyTorch mirror `neurst_pt`
from $NEURST_REFERENCE, the reference checkout or the copy of it oracle/build_ref.py stages under oracle/_ref
(TensorFlow is not installed; SURVEY.md §8c).

It installs a fake `tensorflow` module exposing the few symbols neurst_pt / neurst.utils touch
(tf.nest, tf.io.gfile, tf.errors.OpError), pre-seeds `neurst` / `neurst.utils` as namespace packages so that
neurst/__init__.py (which imports every TF sub-package) is never executed, and stubs `neurst.utils.compat`.
Users: oracle/make_golden.py, the registry plug-in and weight-map tests, bench.py's reference CPU leg.
"""
import importlib
import os
import shutil
import sys
import types

from oracle import build_ref

REF = os.environ.get("NEURST_REFERENCE") or build_ref.reference_root() or ""


def _flatten(x):
    if isinstance(x, (list, tuple)):
        out = []
        for y in x:
            out.extend(_flatten(y))
        return out
    if isinstance(x, dict):
        out = []
        for k in sorted(x):
            out.extend(_flatten(x[k]))
        return out
    return [x]


def _is_nested(x):
    return isinstance(x, (list, tuple, dict))


def _pack_sequence_as(structure, flat):
    it = iter(flat)

    def rec(s):
        if isinstance(s, (list, tuple)):
            return type(s)(rec(y) for y in s)
        if isinstance(s, dict):
            return {k: rec(s[k]) for k in sorted(s)}
        return next(it)
    return rec(structure)


def _map_structure(fn, *structs, **kwargs):
    flats = [_flatten(s) for s in structs]
    return _pack_sequence_as(structs[0], [fn(*a) for a in zip(*flats)])


def install():
    if not os.path.isdir(REF):
        raise RuntimeError("no reference tree: neither NEURST_REFERENCE nor a copy staged by oracle/build_ref.py")
    if "tensorflow" not in sys.modules:
        tf = types.ModuleType("tensorflow")
        nest = types.ModuleType("tensorflow.nest")
        nest.flatten, nest.is_nested = _flatten, _is_nested
        nest.map_structure, nest.pack_sequence_as = _map_structure, _pack_sequence_as
        tf.nest = nest
        io = types.ModuleType("tensorflow.io")
        gfile = types.ModuleType("tensorflow.io.gfile")
        gfile.exists, gfile.isdir, gfile.makedirs = os.path.exists, os.path.isdir, os.makedirs
        gfile.GFile, gfile.copy = open, shutil.copy
        io.gfile = gfile
        tf.io = io
        errors = types.ModuleType("tensorflow.errors")
        errors.OpError = type("OpError", (Exception,), {})
        tf.errors = errors
        tf.Tensor = type("Tensor", (), {})
        sys.modules.update({"tensorflow": tf, "tensorflow.nest": nest, "tensorflow.io": io,
                            "tensorflow.io.gfile": gfile, "tensorflow.errors": errors})
    for name, sub in (("neurst", "neurst"), ("neurst.utils", "neurst/utils")):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [os.path.join(REF, sub)]
            sys.modules[name] = m
    if "neurst.utils.compat" not in sys.modules:
        compat = types.ModuleType("neurst.utils.compat")
        compat.FLOAT_MIN = -1.e9
        compat.CUSTOM_GLOBAL_FLOATX = "float32"
        sys.modules["neurst.utils.compat"] = compat
        sys.modules["neurst.utils"].compat = compat
    if REF not in sys.path:
        sys.path.insert(0, REF)
    return importlib.import_module("neurst_pt")
