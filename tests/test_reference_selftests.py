"""The reference's OWN unit tests (reference tests/test_gantts.py, 5 tests) restated on the oracle port, against what
the unmodified reference computed on the same inputs (tests/golden/selftests.npz, written by make_golden.py, which
also runs those 5 tests on top of the nnmnkwii restatement).  This anchors oracle/nnmnkwii_port.py and the port of
gantts/*.py on the only tests the reference holds for the path (SURVEY.md 8c), at the configurations they use:
In2OutHighwayNet at its default sizes with two windows, T=100, the TTS stream layout 180/3/1/3."""
import os

import numpy as np
import torch

from conftest import GOLDEN, WINDOWS, rel_err
from oracle import gantts_port as gp
from oracle import nnmnkwii_port as nnp

F32_TOL = 2e-6
STREAM_SIZES, HAS_DYNAMIC = [180, 3, 1, 3], [True, True, False, True]
SELECT_CASES = ("1111", "1000", "1001", "0001", "0010", "0100", "1100")
STATIC_CASES = ("1111", "1000", "0100", "1001")


def model_case():
    """Weights and inputs of reference test_model (In2OutHighwayNet(): 118 -> 3 x 512 -> 118, static 59) from a
    numpy RandomState, so that they need not be stored: {state_dict name: array}, x (1,T,118), the mini-batch
    x (B,T,118), y (B,T,59) and lengths (reference tests/test_gantts.py:17-51, batch reduced from 32 to 2)."""
    rs = np.random.RandomState(20)
    sd = {}
    for name, i, o in (("T", 59, 59), ("H.0", 118, 512), ("H.1", 512, 512), ("H.2", 512, 512),
                       ("last_linear", 512, 118)):
        k = 1.0 / np.sqrt(i)
        sd[name + ".weight"] = rs.uniform(-k, k, (o, i)).astype(np.float32)
        sd[name + ".bias"] = rs.uniform(-k, k, o).astype(np.float32)
    T, B = 100, 2
    x1 = rs.rand(1, T, 118).astype(np.float32)
    xb = rs.rand(B, T, 118).astype(np.float32)
    yb = rs.rand(B, T, 59).astype(np.float32)
    lengths = np.array([int(v) for v in rs.randint(50, T - 1, B - 1)] + [T], dtype=np.int64)
    return sd, x1, xb, yb, lengths


def streams(code):
    return [c == "1" for c in code]


def multistream_input():
    return np.random.RandomState(21).rand(2, 100, 187).astype(np.float32)


def static_input():
    return np.random.RandomState(22).rand(2, 10, 187).astype(np.float32)


def test_reference_unit_tests_pass_on_the_port():
    g = np.load(os.path.join(GOLDEN, "selftests.npz"))
    T_ = torch.from_numpy

    # test_model: two windows, default In2OutHighwayNet (eval mode: dropout off), MaskedMSELoss backward
    sd, x1, xb, yb, lengths = model_case()
    gate = (T_(sd["T.weight"]), T_(sd["T.bias"]))
    layers = [(T_(sd["H.%d.weight" % i]), T_(sd["H.%d.bias" % i])) for i in range(3)]
    layers.append((T_(sd["last_linear.weight"]), T_(sd["last_linear.bias"])))
    R = T_(nnp.unit_variance_mlpg_matrix(WINDOWS[:2], 100))
    _, y = gp.in2out_highway_forward(T_(x1), R, gate, layers, static_dim=59)
    assert y.shape == (1, 100, 59)
    assert rel_err(y.numpy(), g["model_y_static"]) < F32_TOL
    x = T_(xb).requires_grad_(True)
    _, y_hat = gp.in2out_highway_forward(x, R, gate, layers, static_dim=59)
    loss = gp.masked_mse(y_hat, T_(yb), lengths=T_(lengths))
    loss.backward()
    assert y_hat.shape == (2, 100, 59)
    assert rel_err(loss.detach().numpy(), g["model_loss"]) < F32_TOL
    assert rel_err(x.grad.numpy(), g["model_grad_x"]) < F32_TOL

    # test_select_streams
    z = torch.zeros(32, 100, 63)
    assert gp.select_streams(z, [60, 1, 1, 1], streams("1111")).size() == (32, 100, 63)
    assert gp.select_streams(z, [60, 1, 1, 1], streams("1000")).size() == (32, 100, 60)
    assert gp.select_streams(z, [60, 1, 1, 1], streams("1001")).size() == (32, 100, 61)
    a = torch.arange(0, 63).expand(2, 3, 63)
    for code in SELECT_CASES:
        got = gp.select_streams(a, [60, 1, 1, 1], streams(code)).numpy()
        assert np.array_equal(got, g["select_" + code]), code
    assert np.array_equal(gp.select_streams(a, [60, 1, 1, 1], streams("0001")).squeeze(-1), a[:, :, -1])
    assert np.array_equal(gp.select_streams(a, [60, 1, 1, 1], streams("0100")).squeeze(-1), a[:, :, -3])

    # test_get_static_stream_sizes
    sizes = gp.get_static_stream_sizes(STREAM_SIZES, HAS_DYNAMIC, 3)
    assert np.array_equal(sizes, [60, 1, 1, 1]) and np.array_equal(sizes, g["static_stream_sizes"])

    # test_get_static_features
    s = T_(static_input())
    for code, width in zip(STATIC_CASES, (63, 60, 1, 61)):
        got = gp.get_static_features(s, 3, STREAM_SIZES, HAS_DYNAMIC, streams=streams(code))
        assert got.shape == (2, 10, width)
        assert np.array_equal(got.numpy(), g["static_" + code]), code

    # test_multi_stream_mlpg: the per-stream MLPG results are the unit-variance MLPG of the stream, vuv copied
    m = T_(multistream_input())
    R = T_(nnp.unit_variance_mlpg_matrix(WINDOWS, 100))
    y = gp.multi_stream_mlpg(m, R, STREAM_SIZES, HAS_DYNAMIC)
    assert y.shape == (2, 100, 63)
    assert rel_err(y.numpy(), g["mlpg_y"]) < F32_TOL
    assert torch.equal(nnp.unit_variance_mlpg(R, m[:, :, :180]), y[:, :, :60])
    assert torch.equal(nnp.unit_variance_mlpg(R, m[:, :, 180:183]).squeeze(-1), y[:, :, 60])
    assert torch.equal(m[:, :, 183], y[:, :, 61])
    assert torch.equal(nnp.unit_variance_mlpg(R, m[:, :, 184:187]).squeeze(-1), y[:, :, 62])
    assert gp.get_static_features(m, 3, STREAM_SIZES, HAS_DYNAMIC).size() == y.size()
