"""CPU-only tests: C-ABI library loads and exports every declared symbol, host-side logic
(stream column tables, MLPG table, argument validation), and the no-CPU-fallback rule."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, WINDOWS
from oracle import nnmnkwii_port as nnp


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from gantts_b200 import _lib
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from gantts_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gantts_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(gantts_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), "libgantts_b200.so does not export %s" % name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.gantts_version() >= 100
    assert lib.gantts_last_error_string() is not None


def test_library_is_sm100a_only(lib):
    import subprocess
    from gantts_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out


def test_mlpg_table_matches_dense_inverse(lib):
    from gantts_b200 import ops
    for wins, T in ((WINDOWS, 64), (WINDOWS, 257), (WINDOWS[:2], 50), (WINDOWS[:1], 9), (WINDOWS, 3)):
        tab = ops.mlpg_table_host(wins, T)
        Pi = np.linalg.inv(nnp.normal_matrix(wins, T))
        K = 24
        for t in range(T):
            for j in range(49):
                c = t + j - K
                exp = Pi[t, c] if 0 <= c < T else 0.0
                assert abs(tab[t, j] - exp) < 2e-7


def test_mlpg_table_cholesky_rows_solve_the_normal_equations():
    """Columns 52..59 of the table = rows of the banded Cholesky factor L of P = W^T W (1/L_tt, L[t][t-1], L[t][t-2] and the
    transposed entries L[t+1][t], L[t+2][t]).  The substitution the round-2 MLPG kernels run (forward with the first three,
    backward with the transposed pair), evaluated here in numpy from the library's own table, solves P y = b -- on the whole
    sequence and, with the kernels' 28-frame warm-up from a zero state, on a 32-frame chunk in the middle."""
    from gantts_b200 import ops
    rng = np.random.default_rng(1)
    for wins, T in ((WINDOWS, 200), (WINDOWS[:2], 77), (WINDOWS, 5), (WINDOWS[:1], 9)):
        tab = ops.mlpg_table_full_host(wins, T).astype(np.float64)
        P = nnp.normal_matrix(wins, T)
        L = np.zeros((T, T))
        for t in range(T):
            L[t, t] = 1.0 / tab[t, 52]
            if t >= 1:
                L[t, t - 1] = tab[t, 53]
            if t >= 2:
                L[t, t - 2] = tab[t, 54]
            if t + 1 < T:
                assert abs(tab[t, 56] - tab[t + 1, 53]) < 1e-12          # L[t+1][t] stored twice
            if t + 2 < T:
                assert abs(tab[t, 57] - tab[t + 2, 54]) < 1e-12
        assert np.abs(L @ L.T - P).max() < 2e-6 * np.abs(P).max()

        def solve(b, s, e):
            """forward then backward substitution over rows [s, e) from a zero state, table rows as the kernels read them"""
            z = np.zeros(T)
            z1 = z2 = 0.0
            for t in range(s, e):
                z[t] = (b[t] - tab[t, 53] * z1 - tab[t, 54] * z2) * tab[t, 52]
                z2, z1 = z1, z[t]
            y = np.zeros(T)
            y1 = y2 = 0.0
            for t in range(e - 1, s - 1, -1):
                y[t] = (z[t] - tab[t, 56] * y1 - tab[t, 57] * y2) * tab[t, 52]
                y2, y1 = y1, y[t]
            return y
        b = rng.standard_normal(T)
        ref = np.linalg.solve(P, b)
        assert np.abs(solve(b, 0, T) - ref).max() < 5e-6 * np.abs(ref).max()
        if T >= 120:
            t0, t1, sw = 80, 112, 28
            y = solve(b, t0 - sw, t1 + sw)
            assert np.abs(y[t0:t1] - ref[t0:t1]).max() < 5e-6 * np.abs(ref).max()


def test_mlpg_table_fir_equals_dense_R():
    """Stencil + truncated FIR (the CUDA algorithm, evaluated here in numpy from the library's own
    table) reproduces the reference's dense R matmul."""
    from gantts_b200 import ops
    T, sd = 120, 5
    rng = np.random.default_rng(0)
    mu = rng.standard_normal((T, 3 * sd))
    R = nnp.unit_variance_mlpg_matrix(WINDOWS, T).astype(np.float64)
    ref = R @ np.vstack([mu[:, w * sd:(w + 1) * sd] for w in range(3)])
    tab = ops.mlpg_table_host(WINDOWS, T).astype(np.float64)
    b = np.zeros((T, sd))
    for w, (l, u, coef) in enumerate(WINDOWS):
        for k in range(-l, u + 1):
            for t in range(T):
                if 0 <= t - k < T:
                    b[t] += coef[k + l] * mu[t - k, w * sd:(w + 1) * sd]
    y = np.zeros((T, sd))
    for t in range(T):
        for j in range(49):
            c = t + j - 24
            if 0 <= c < T:
                y[t] += tab[t, j] * b[c]
    assert np.max(np.abs(y - ref)) / np.max(np.abs(ref)) < 1e-6


def test_bad_windows_rejected(lib):
    from gantts_b200 import _lib
    w = _lib.make_windows([(0, 0, [1.0])])
    w.n = 9
    tab = np.zeros((4, 49), np.float32)
    assert lib.gantts_mlpg_table(ctypes.byref(w), 4, tab.ctypes.data) == 1
    assert b"window" in lib.gantts_last_error_string()
    with pytest.raises(RuntimeError):
        _lib.make_windows([(3, 3, [1.0] * 7)])


def test_stream_column_tables(golden_ops):
    from gantts_b200 import multistream as ms
    assert np.array_equal(ms.get_static_stream_sizes([180, 3, 1, 3], [True, True, False, True], 3),
                          golden_ops["static_sizes"])
    x = np.arange(63)
    for name in ("1111", "1000", "1001", "0010", "0101"):
        cols = ms.select_stream_columns([60, 1, 1, 1], [c == "1" for c in name])
        assert np.array_equal(x[cols], golden_ops["select_" + name][0, 0])
    y = golden_ops["ms_in"]
    cols = ms.static_feature_columns(3, [180, 3, 1, 3], [True, True, False, True], [True] * 4)
    assert np.array_equal(y[:, :, cols], golden_ops["static_all"])
    cols = ms.static_feature_columns(3, [180, 3, 1, 3], [True, True, False, True], [True, False, False, True])
    assert np.array_equal(y[:, :, cols], golden_ops["static_1001"])
    entries, n = ms.mlpg_stream_entries([180, 3, 1, 3], [True, True, False, True], [True] * 4, 3)
    assert entries == [(0, 60, True, 0), (180, 1, True, 60), (183, 1, False, 61), (184, 1, True, 62)] and n == 63
    entries, n = ms.mlpg_stream_entries([180, 3, 1, 3], [True, True, False, True], [True, False, True, False], 3)
    assert entries == [(0, 60, True, 0), (183, 1, False, 60)] and n == 61


def test_no_cpu_fallback(lib):
    """CPU tensors are rejected loudly instead of being routed to a host implementation."""
    import gantts_b200
    from gantts_b200 import ops
    x = torch.zeros(2, 5, 63)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gantts_b200.multistream.select_streams(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gantts_b200.seqloss.sequence_mask(torch.LongTensor([3, 2]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gantts_b200.models.MLP(4, 2)(torch.zeros(3, 4))
    with pytest.raises(RuntimeError):
        gantts_b200.seqloss.MaskedMSELoss()(x, x)
    with pytest.raises(RuntimeError, match="dimention"):
        gantts_b200.multistream.multi_stream_mlpg(torch.zeros(1, 4, 100), None)
    assert ops.windows_for(3)[2] == (1, 1, (1.0, -2.0, 1.0))


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under gantts_b200/ may reference it."""
    pkg = os.path.join(ROOT, "gantts_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src, os.path.join(dirpath, f)


def test_state_dict_keys_match_reference_layout():
    import gantts_b200
    m = gantts_b200.models.MLP(in_dim=7, out_dim=3, num_hidden=2, hidden_dim=5)
    assert list(m.state_dict()) == ["layers.0.weight", "layers.0.bias", "layers.1.weight", "layers.1.bias",
                                    "last_linear.weight", "last_linear.bias"]
    h = gantts_b200.models.In2OutHighwayNet(in_dim=6, out_dim=6, static_dim=2, num_hidden=2, hidden_dim=4)
    assert list(h.state_dict()) == ["T.weight", "T.bias", "H.0.weight", "H.0.bias", "H.1.weight", "H.1.bias",
                                    "last_linear.weight", "last_linear.bias"]
    assert h.include_parameter_generation() and not m.include_parameter_generation()


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """Without the built .so every op raises (no silent eager/CPU route)."""
    from gantts_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libgantts_b200.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()
    # an existing file that lacks a declared symbol is rejected too
    import ctypes.util
    libm = ctypes.util.find_library("m")
    if libm:
        monkeypatch.setattr(_lib, "LIB_PATH", ctypes.CDLL(libm)._name if os.path.isabs(ctypes.CDLL(libm)._name)
                            else "/usr/lib/x86_64-linux-gnu/" + libm)
        if os.path.exists(_lib.LIB_PATH):
            with pytest.raises(AttributeError):
                _lib.load()


def test_distortion_struct_matches_header():
    """ctypes mirror of gantts_distortion_cols_t: same field order as include/gantts_b200.h."""
    from gantts_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gantts_b200.h")).read()
    body = hdr[hdr.index("typedef struct {\n  int mcd_start"):hdr.index("} gantts_distortion_cols_t;")]
    names = [tok.strip(" ;") for line in body.splitlines()[1:] for tok in line.replace("int ", "").split(",") if tok.strip(" ;")]
    assert names == [f for f, _ in _lib.DistortionColsT._fields_]


def test_gan_step_struct_layout_matches_header(tmp_path):
    """ctypes mirror of gantts_gan_step_t against the C compiler's view of include/gantts_b200.h: total size and the
    offsets of the first / middle / last fields (incl. the optimiser block appended in round 2)."""
    import ctypes
    import subprocess
    from gantts_b200 import _lib
    fields = ["B", "g", "d", "g_sumW", "streams", "windows", "mlpg_table", "n_static", "static_cols", "adv_cols", "lr_g", "adv_w",
              "optimizer", "beta1", "opt_step", "g_sqW", "d_sqb"]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gantts_b200.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(gantts_gan_step_t));\n' +
                   "".join('  printf(" %%zu", offsetof(gantts_gan_step_t, %s));\n' % f for f in fields) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    want = [ctypes.sizeof(_lib.GanStepT)] + [getattr(_lib.GanStepT, f).offset for f in fields]
    assert got == want


def test_dropout_hash_statistics():
    """The counter-hash keep mask (tests/dropout_mirror.py = csrc/common.cuh bit for bit; the GPU suite pins the kernels to
    the mirror): keep rate, independence of the four fields of a quad / of neighbouring quads / of neighbouring rows, and
    binomial dispersion of the per-column and per-row keep rates."""
    import dropout_mirror as dm
    rows, n = 8192, 256
    for seed, p in ((12345678901234567, 0.5), (4242 * 4 + 1, 0.2), (99, 0.5)):
        m = dm.keep_mask(seed, rows, n, p).astype(np.float64)
        assert abs(m.mean() - (1.0 - p)) < 2e-3
        z = m - m.mean()

        def corr(a, b):
            return float((a * b).mean() / np.sqrt((a * a).mean() * (b * b).mean()))
        pairs = [(z[:, 0::4], z[:, 1::4]), (z[:, 0::4], z[:, 2::4]), (z[:, 0::4], z[:, 3::4]), (z[:, 1::4], z[:, 2::4]),
                 (z[:, 2::4], z[:, 3::4]), (z[:, :-4], z[:, 4:]), (z[:-1], z[1:])]
        assert max(abs(corr(a, b)) for a, b in pairs) < 8e-3          # 1/sqrt(samples) = 1.4e-3
        q = p * (1.0 - p)
        assert abs(m.mean(0).std() / np.sqrt(q / rows) - 1.0) < 0.25
        assert abs(m.mean(1).std() / np.sqrt(q / n) - 1.0) < 0.1
    assert not dm.keep_mask(7, 64, 64, 1.0).any() and dm.keep_mask(7, 64, 64, 0.0).all()


def test_bench_algorithmic_work_matches_survey_8d():
    """bench.py's roofline numerator: SURVEY.md 8(d) algorithmic MACs per padded frame of the de-duplicated GAN step --
    cfg2 3 449 856 (= 3 F_G - k0 + 8 F_D - 256 d_in); cfg3 / cfg5: 3 x (LSTM stack 15.41 M / 16.42 M + hidden2out
    181 248 / 191 488) minus the first layer's input-gradient product, plus the discriminator's share."""
    import bench
    assert bench.algorithmic_flops_per_frame(bench.WORKLOADS["cfg2"]) == 2.0 * 3449856
    for name, lstm_macs, out_macs in (("cfg3", 15405056, 181248), ("cfg5", 16420864, 191488)):
        w = bench.WORKLOADS[name]
        H, F_L, inp = w["g_hidden"], 0, w["d_in"]
        for _ in range(w["g_layers"]):
            F_L += 2 * 4 * H * (inp + H)
            inp = 2 * H
        assert F_L == lstm_macs and 2 * H * w["d_out"] == out_macs
        dd = w["d_dims"]
        F_D = sum(a * b for a, b in zip(dd[:-1], dd[1:]))
        want = 3 * (F_L + out_macs) - 2 * 4 * H * w["d_in"] + 2 * w.get("static_dim", 0) ** 2 + 8 * F_D - dd[1] * dd[0]
        assert bench.algorithmic_flops_per_frame(w) == 2.0 * want


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole, large ones as a seeded sample of their elements, the
    directory stays within the budget, and the same shapes always sample the same elements."""
    import bench
    rs = np.random.RandomState(0)
    arrays = {"loss_g": np.float32(rs.rand(1)), "y_hat": rs.rand(600, 187).astype(np.float32),
              "g.w": rs.rand(512, 425).astype(np.float32), "d.b": rs.rand(256).astype(np.float64)}
    budget = 1 << 19
    for run in ("a", "b"):
        bench.dump_outputs(arrays, str(tmp_path / run), budget=budget)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["d.b.npy", "g.w.npy", "loss_g.npy", "y_hat.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= budget
    for name, a in arrays.items():
        got, again = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert got.dtype == a.dtype and np.array_equal(got, again)
        if name in ("loss_g", "d.b"):
            assert np.array_equal(got, a)
        else:
            assert got.ndim == 1 and 0 < got.size < a.size and np.isin(got, a.reshape(-1)).all()
