"""Import the UNMODIFIED reference Python (r9y9/gantts) from /root/reference.  TEST INFRASTRUCTURE.

Only usable where the reference tree is present (``GANTTS_REFERENCE_ROOT``); it is what
``tests/golden/make_golden.py`` uses to generate the committed golden vectors.  The tests read
only those vectors, so they run without the reference.

The reference does not import as shipped (SURVEY.md section 8c): ``gantts/__init__.py:4`` needs
a generated ``gantts/version.py`` (setup.py:24-36), ``multistream.py:11-12``/``models.py:8``
import nnmnkwii, ``hparams.py:3`` imports tensorflow 1.x, ``train.py:24,44`` import docopt and
tensorboard_logger.  The loader registers in-memory stand-ins for exactly those names (the
nnmnkwii arithmetic comes from ``oracle.nnmnkwii_port``) and then executes the reference files
where they lie.  No reference source is copied.
"""
import ast
import importlib.util
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("GANTTS_REFERENCE_ROOT", "/root/reference")
_PREFIX = "_refgantts"


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "gantts", "models.py"))


class _HParams(object):
    """Minimal stand-in for tf.contrib.training.HParams (reference hparams.py:3,16)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def values(self):
        return dict(self.__dict__)

    def parse(self, s):
        for item in [p for p in s.split(",") if p.strip()]:
            k, v = item.split("=", 1)
            try:
                v = ast.literal_eval(v)
            except Exception:
                pass
            setattr(self, k.strip(), v)
        return self


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    return m


def _stub_modules():
    from . import nnmnkwii_port as nn_port
    mods = {}
    nnm = _module("nnmnkwii")
    nnm.paramgen = _module("nnmnkwii.paramgen",
                           unit_variance_mlpg_matrix=nn_port.unit_variance_mlpg_matrix)
    nnm.autograd = _module("nnmnkwii.autograd", unit_variance_mlpg=nn_port.unit_variance_mlpg)
    nnm.preprocessing = _module("nnmnkwii.preprocessing", delta_features=nn_port.delta_features)
    nnm.metrics = _module("nnmnkwii.metrics")
    nnm.datasets = _module("nnmnkwii.datasets", FileSourceDataset=object, FileDataSource=object,
                           MemoryCacheDataset=object)
    for sub in ("paramgen", "autograd", "preprocessing", "metrics", "datasets"):
        mods["nnmnkwii." + sub] = getattr(nnm, sub)
    mods["nnmnkwii"] = nnm
    tf = _module("tensorflow")
    tf.contrib = _module("tensorflow.contrib")
    tf.contrib.training = _module("tensorflow.contrib.training", HParams=_HParams)
    mods["tensorflow"] = tf
    mods["tensorflow.contrib"] = tf.contrib
    mods["tensorflow.contrib.training"] = tf.contrib.training
    mods["docopt"] = _module("docopt", docopt=lambda *a, **k: {})
    mods["tensorboard_logger"] = _module("tensorboard_logger", configure=lambda *a, **k: None,
                                         log_value=lambda *a, **k: None)
    return mods


def _exec_file(modname, path, package=None):
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    if package is not None:
        mod.__package__ = package
    sys.modules[modname] = mod
    spec.loader.exec_module(mod)
    return mod


class Reference(object):
    """Handle on the imported reference modules: ``.models .multistream .seqloss .train .hparams``."""


_cached = None


def load(with_train=True):
    """Execute the reference files under temporary ``sys.modules`` bindings and return them.

    The bindings for ``gantts``/``nnmnkwii``/``tensorflow``/... are removed again afterwards so
    that the product package ``gantts`` (the drop-in alias of ``gantts_b200``) is never shadowed.
    """
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    if not hasattr(np, "int"):
        np.int = int            # reference train.py:148 uses the removed alias
    stubs = _stub_modules()
    touched = list(stubs) + ["gantts", "gantts.version", "gantts.models", "gantts.multistream",
                             "gantts.seqloss", "hparams", "train"]
    saved = {k: sys.modules.get(k) for k in touched}
    ref = Reference()
    try:
        sys.modules.update(stubs)
        pkg = types.ModuleType("gantts")
        pkg.__path__ = [os.path.join(REFERENCE_ROOT, "gantts")]
        sys.modules["gantts"] = pkg
        sys.modules["gantts.version"] = _module("gantts.version", __version__="0.1.1")
        g = os.path.join(REFERENCE_ROOT, "gantts")
        ref.multistream = _exec_file("gantts.multistream", os.path.join(g, "multistream.py"), "gantts")
        ref.seqloss = _exec_file("gantts.seqloss", os.path.join(g, "seqloss.py"), "gantts")
        ref.models = _exec_file("gantts.models", os.path.join(g, "models.py"), "gantts")
        pkg.models, pkg.multistream, pkg.seqloss = ref.models, ref.multistream, ref.seqloss
        if with_train:
            ref.hparams = _exec_file("hparams", os.path.join(REFERENCE_ROOT, "hparams.py"))
            ref.train = _exec_file("train", os.path.join(REFERENCE_ROOT, "train.py"))
            ref.train.use_cuda = False
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    _cached = ref
    return ref
