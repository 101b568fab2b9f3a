"""CPU tests of the import shims that let the reference's train.py / hparams.py run unchanged on this image."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, WINDOWS
from oracle import nnmnkwii_port as nnp

COMPAT = os.path.join(ROOT, "compat")


@pytest.fixture(scope="module", autouse=True)
def _path():
    import __graft_entry__
    __graft_entry__.build()
    sys.path.insert(1, COMPAT)
    yield
    sys.path.remove(COMPAT)


def test_unit_variance_mlpg_matrix_shim_matches_dense_definition():
    from nnmnkwii.paramgen import unit_variance_mlpg_matrix
    for wins, T in ((WINDOWS, 7), (WINDOWS, 100), (WINDOWS[:2], 40), (WINDOWS[:1], 6)):
        a, b = unit_variance_mlpg_matrix(wins, T), nnp.unit_variance_mlpg_matrix(wins, T)
        assert a.shape == b.shape and a.dtype == np.float32
        assert np.abs(a - b).max() < 2e-7
    assert unit_variance_mlpg_matrix(WINDOWS, 100) is unit_variance_mlpg_matrix(WINDOWS, 100)   # memoised


def test_delta_features_and_scaling_shims():
    from nnmnkwii import preprocessing as P
    x = np.random.RandomState(0).randn(9, 3)
    assert np.allclose(P.delta_features(x, WINDOWS), nnp.delta_features(x, WINDOWS))
    mn, mx = x.min(0), x.max(0)
    m_, s_ = P.minmax_scale_params(mn, mx, feature_range=(0.01, 0.99))
    y = P.minmax_scale(x, min_=m_, scale_=s_, feature_range=(0.01, 0.99))
    assert np.allclose(y.min(0), 0.01) and np.allclose(y.max(0), 0.99)
    mean, var = P.meanvar([x, 2 * x])
    allx = np.vstack([x, 2 * x])
    assert np.allclose(mean, allx.mean(0)) and np.allclose(var, allx.var(0))
    assert np.allclose(P.inv_scale(P.scale(x, mean, np.sqrt(var)), mean, np.sqrt(var)), x)


def test_metrics_shims():
    from nnmnkwii import metrics
    rs = np.random.RandomState(1)
    X, Y = rs.randn(2, 5, 4), rs.randn(2, 5, 4)
    lens = [5, 3]
    exp = 10 / np.log(10) * np.sqrt(2) * (np.sqrt(((X[0] - Y[0]) ** 2).sum(-1)).sum() +
                                          np.sqrt(((X[1, :3] - Y[1, :3]) ** 2).sum(-1)).sum()) / 8
    assert abs(metrics.melcd(X, Y, lens) - exp) < 1e-9
    v1 = np.array([[1, 1, 0, 1, 1], [1, 0, 1, 1, 1]], float)
    v2 = np.array([[1, 0, 0, 1, 1], [1, 1, 1, 0, 0]], float)
    assert metrics.vuv_error(v1, v2, lens) == 2 / 8
    f1, f2 = rs.rand(2, 5, 1), rs.rand(2, 5, 1)
    both = [(0, 0), (0, 3), (0, 4), (1, 0), (1, 2)]
    exp = sum((f1[b, t, 0] - f2[b, t, 0]) ** 2 for b, t in both) / len(both)
    assert abs(metrics.lf0_mean_squared_error(f1, v1, f2, v2, lens) - exp) < 1e-12
    with pytest.raises(ZeroDivisionError):
        metrics.lf0_mean_squared_error(f1, v1 * 0, f2, v2, lens)


def test_hparams_and_docopt_shims():
    from tensorflow.contrib.training import HParams
    hp = HParams(a=1, b=[1, 2], name="x", d={"k": None})
    hp.parse('a=5,b=[3,4,5],d={"k": 7, "j": [1,2]}')
    assert (hp.a, hp.b, hp.d) == (5, [3, 4, 5], {"k": 7, "j": [1, 2]}) and hp.values()["name"] == "x"
    with pytest.raises(ValueError):
        hp.parse("nope=1")
    from docopt import docopt
    doc = """usage: t.py [options] <in> <out>

options:
    --w_d=<f>   weight [default: 1.0].
    --flag      a flag.
    -h, --help  help
"""
    args = docopt(doc, ["--w_d", "0.5", "a", "b"])
    assert args == {"--w_d": "0.5", "--flag": False, "--help": False, "<in>": "a", "<out>": "b"}
    assert docopt(doc, ["--flag", "a", "b"])["--w_d"] == "1.0"


_RESOLVE_IMPORTS = r"""
import importlib, json, sys
sys.path[:0] = [ROOT, COMPAT]
g = json.load(open(GOLDEN))
where = {}
for imp in g["imports"]:
    if imp["module"] == "hparams":        # the reference's own configuration file, next to its train.py
        continue
    mod = importlib.import_module(imp["module"])
    for name in imp["names"]:
        obj = getattr(mod, name, None)
        if obj is None:
            obj = importlib.import_module(imp["module"] + "." + name)
        where[imp["module"] + ":" + name] = getattr(obj, "__module__", None) or obj.__name__
    where[imp["module"]] = getattr(mod, "__file__", None) or ""
import gantts, tensorflow
models = {"%s.%s" % (cfg, role): getattr(gantts.models, name).__module__
          for cfg, roles in g["models"].items() for role, name in roles.items()}
print(json.dumps({"gantts": gantts.__name__, "where": where, "models": models,
                  "hparams_class": tensorflow.contrib.training.HParams.__module__}))
"""


def test_reference_train_py_imports_unchanged_on_the_alias_package():
    """Every module-level import of the reference's train.py and hparams.py (recorded from the unmodified files in
    tests/golden/trainpy_imports.json) resolves with PYTHONPATH = repo : repo/compat, in a fresh interpreter: the
    gantts.* names to the B200 package, nnmnkwii / tensorflow / docopt / tensorboard_logger to the shims, and the
    generator / discriminator classes hparams.py names are found in gantts.models."""
    golden = os.path.join(ROOT, "tests", "golden", "trainpy_imports.json")
    code = "ROOT, COMPAT, GOLDEN = %r, %r, %r\n" % (ROOT, COMPAT, golden) + _RESOLVE_IMPORTS
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    got = json.loads(out.stdout.strip().splitlines()[-1])
    assert got["gantts"] == "gantts"
    recorded = json.load(open(golden))
    assert {"vc", "tts_duration", "tts_acoustic"} <= set(recorded["models"])
    assert recorded["models"]["vc"]["generator"] == "In2OutHighwayNet"
    assert set(got["models"].values()) == {"gantts_b200.models"}, got["models"]
    assert got["hparams_class"].startswith("tensorflow.")
    w = got["where"]
    assert w["gantts.seqloss:MaskedMSELoss"] == "gantts_b200.seqloss"
    assert w["nnmnkwii.paramgen:unit_variance_mlpg_matrix"] == "nnmnkwii.paramgen"
    for key, module in w.items():
        name = key.split(":")[0]
        if ":" in key and name.startswith("gantts"):
            assert module.startswith("gantts_b200."), (key, module)
        if ":" not in key and name.split(".")[0] in ("nnmnkwii", "tensorflow", "docopt", "tensorboard_logger"):
            assert os.path.realpath(module).startswith(os.path.realpath(COMPAT) + os.sep), (key, module)
