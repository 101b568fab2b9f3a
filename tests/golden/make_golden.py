"""Generate tests/golden/*.npz by running the UNMODIFIED reference (r9y9/gantts @ fb1e75f, imported
read-only from /root/reference through oracle.reference_loader) on seeded inputs.

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Everything stored is produced by the reference's own code paths -- gantts/models.py,
gantts/multistream.py, gantts/seqloss.py and the step functions of train.py (apply_generator,
update_discriminator, update_generator) -- on top of the nnmnkwii restatement in
oracle/nnmnkwii_port.py (nnmnkwii itself is not installable offline: "parity unpinned" for that
third-party arithmetic, see oracle/__init__.py).  Inputs and weights are stored next to the
outputs so the tests do not depend on torch's RNG stream staying stable across versions.
"""
import json
import os
import sys

import numpy as np
import torch
from torch import optim

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import reference_loader  # noqa: E402
from oracle import nnmnkwii_port as nnp  # noqa: E402

WINDOWS = [
    (0, 0, np.array([1.0])),
    (1, 1, np.array([-0.5, 0.0, 0.5])),
    (1, 1, np.array([1.0, -2.0, 1.0])),
]


def npy(t):
    return t.detach().cpu().numpy().copy()


def lengths_desc(rng, B, T):
    ls = sorted([T] + [int(v) for v in rng.integers(T // 2, T, B - 1)], reverse=True)
    return ls


def gen_seqloss(ref, out):
    rng = np.random.default_rng(11)
    B, T, D = 5, 23, 7
    lengths = torch.LongTensor(lengths_desc(rng, B, T))
    out["mask_lengths"] = lengths.numpy()
    out["mask"] = npy(ref.seqloss.sequence_mask(lengths))
    out["mask_maxlen30"] = npy(ref.seqloss.sequence_mask(lengths, 30))
    a = torch.randn(B, T, D, requires_grad=True)
    b = torch.randn(B, T, D)
    crit = ref.seqloss.MaskedMSELoss()
    loss = crit(a, b, lengths=lengths)
    loss.backward()
    out["mse_in"], out["mse_tgt"] = npy(a), npy(b)
    out["mse_loss"], out["mse_grad"] = npy(loss), npy(a.grad)
    m = ref.seqloss.sequence_mask(lengths).unsqueeze(-1)
    out["mse_loss_mask"] = npy(crit(a, b, mask=m))


def gen_multistream(ref, out):
    ms = ref.multistream
    x = torch.arange(0, 63).float().expand(2, 4, 63)
    for name, streams in [("1111", [1, 1, 1, 1]), ("1000", [1, 0, 0, 0]), ("1001", [1, 0, 0, 1]),
                          ("0010", [0, 0, 1, 0]), ("0101", [0, 1, 0, 1])]:
        out["select_" + name] = npy(ms.select_streams(x, [60, 1, 1, 1], [bool(s) for s in streams]))
    out["static_sizes"] = ms.get_static_stream_sizes([180, 3, 1, 3], [True, True, False, True], 3)
    torch.manual_seed(5)
    B, T = 3, 37
    y = torch.randn(B, T, 187)
    out["ms_in"] = npy(y)
    out["static_all"] = npy(ms.get_static_features(y, 3, [180, 3, 1, 3], [True, True, False, True]))
    out["static_1001"] = npy(ms.get_static_features(y, 3, [180, 3, 1, 3], [True, True, False, True],
                                                    streams=[True, False, False, True]))
    from oracle.nnmnkwii_port import unit_variance_mlpg_matrix
    R = torch.from_numpy(unit_variance_mlpg_matrix(WINDOWS, T))
    yv = y.clone().requires_grad_(True)
    z = ms.multi_stream_mlpg(yv, R, [180, 3, 1, 3], [True, True, False, True])
    g = torch.randn_like(z)
    z.backward(g)
    out["mlpg_out"], out["mlpg_gout"], out["mlpg_gin"] = npy(z), npy(g), npy(yv.grad)
    z2 = ms.multi_stream_mlpg(y, R, [180, 3, 1, 3], [True, True, False, True],
                              streams=[True, False, True, False])
    out["mlpg_out_1010"] = npy(z2)
    # VC layout: a single dynamic stream 59*3
    v = torch.randn(2, 50, 177)
    Rv = torch.from_numpy(unit_variance_mlpg_matrix(WINDOWS, 50))
    from oracle.nnmnkwii_port import unit_variance_mlpg
    out["vc_in"], out["vc_out"] = npy(v), npy(unit_variance_mlpg(Rv, v))
    # two-window case of reference tests/test_gantts.py:18-21
    w2 = WINDOWS[:2]
    v2 = torch.randn(2, 20, 10)
    R2 = torch.from_numpy(unit_variance_mlpg_matrix(w2, 20))
    out["w2_in"], out["w2_out"] = npy(v2), npy(unit_variance_mlpg(R2, v2))


def state_arrays(model, prefix, out):
    for k, v in model.state_dict().items():
        out[prefix + k] = npy(v)


def gen_models(ref, out):
    torch.manual_seed(7)
    M = ref.models
    g = M.MLP(in_dim=20, out_dim=187, num_hidden=3, hidden_dim=32, dropout=0.5, last_sigmoid=False)
    d = M.MLP(in_dim=58, out_dim=1, num_hidden=3, hidden_dim=16, dropout=0.5, last_sigmoid=True)
    g.eval(), d.eval()
    x = torch.rand(3, 11, 20, requires_grad=True)
    yg = g(x)
    gy = torch.randn_like(yg)
    yg.backward(gy)
    state_arrays(g, "mlpg_", out)
    out["mlp_g_x"], out["mlp_g_y"], out["mlp_g_gy"], out["mlp_g_gx"] = npy(x), npy(yg), npy(gy), npy(x.grad)
    for k, p in g.named_parameters():
        out["mlp_g_grad_" + k] = npy(p.grad)
    xd = torch.randn(3, 11, 58)
    state_arrays(d, "mlpd_", out)
    out["mlp_d_x"], out["mlp_d_y"] = npy(xd), npy(d(xd))
    # In2OutHighwayNet (VC), eval mode
    from oracle.nnmnkwii_port import unit_variance_mlpg_matrix
    h = M.In2OutHighwayNet(in_dim=30, out_dim=30, static_dim=10, num_hidden=2, hidden_dim=24, dropout=0.5)
    h.eval()
    xh = torch.randn(2, 17, 30)
    R = torch.from_numpy(unit_variance_mlpg_matrix(WINDOWS, 17))
    yh, ys = h(xh, R)
    state_arrays(h, "hw_", out)
    out["hw_x"], out["hw_y"], out["hw_ystatic"] = npy(xh), npy(yh), npy(ys)
    # LSTMRNN (bidirectional, 2 layers), eval mode, ragged lengths
    l = M.LSTMRNN(in_dim=12, out_dim=9, num_hidden=2, hidden_dim=16, bidirectional=True, dropout=0.0)
    l.eval()
    xl = torch.randn(3, 14, 12)
    lens = [14, 9, 6]
    for b, n in enumerate(lens):
        xl[b, n:] = 0
    yl = l(xl, lens)
    state_arrays(l, "lstm_", out)
    out["lstm_x"], out["lstm_y"], out["lstm_lengths"] = npy(xl), npy(yl), np.array(lens)


def gen_step(ref, out, cond, tag):
    """Two consecutive mini-batches through the reference's own step functions (train.py:336-355,
    245-279, 282-320) with dropout p=0 so train mode is deterministic; Adagrad as in
    hparams.py:223-227,240-244."""
    tr, hparams = ref.train, ref.hparams
    hp = hparams.tts_acoustic
    hp.discriminator_linguistic_condition = cond
    tr.hp = hp
    torch.manual_seed(21 + int(cond))
    rng = np.random.default_rng(3)
    B, T, Din = 4, 30, 20
    M = ref.models
    g = M.MLP(in_dim=Din, out_dim=187, num_hidden=3, hidden_dim=32, dropout=0.0, last_sigmoid=False)
    d = M.MLP(in_dim=58 + (Din if cond else 0), out_dim=1, num_hidden=3, hidden_dim=16, dropout=0.0,
              last_sigmoid=True)
    state_arrays(g, tag + "g0_", out)
    state_arrays(d, tag + "d0_", out)
    og = optim.Adagrad(g.parameters(), lr=0.01, weight_decay=1e-7)
    od = optim.Adagrad(d.parameters(), lr=0.01, weight_decay=1e-7)
    from oracle.nnmnkwii_port import unit_variance_mlpg_matrix
    R = torch.from_numpy(unit_variance_mlpg_matrix(hp.windows, T))
    g.train(), d.train()
    for it in range(2):
        lens = lengths_desc(rng, B, T)
        x = torch.rand(B, T, Din) * 0.98 + 0.01
        y = torch.randn(B, T, 187)
        for b, n in enumerate(lens):
            x[b, n:] = 0
            y[b, n:] = 0
        lengths = torch.LongTensor(lens)
        y_static = ref.multistream.get_static_features(y, len(hp.windows), hp.stream_sizes,
                                                       hp.has_dynamic_features)
        mask = ref.seqloss.sequence_mask(lengths).unsqueeze(-1)
        og.zero_grad(), od.zero_grad()
        y_hat, y_hat_static = tr.apply_generator(g, x, R, lens)
        ld, lf, lr_, rc, fc = tr.update_discriminator(d, od, x, y_static, y_hat_static, lens, mask, "train")
        lmse, lmge, ladv, lg = tr.update_generator(g, d, og, x, y, y_hat, y_static, y_hat_static,
                                                    1.0, lens, mask, "train", mse_w=0.0, mge_w=1.0)
        p = "%sit%d_" % (tag, it)
        out[p + "x"], out[p + "y"], out[p + "lengths"] = npy(x), npy(y), np.array(lens)
        out[p + "y_hat"], out[p + "y_hat_static"] = npy(y_hat), npy(y_hat_static)
        out[p + "losses"] = np.array([ld, lf, lr_, lmse, lmge, ladv, lg], dtype=np.float64)
        out[p + "counts"] = np.array([rc, fc], dtype=np.float64)
        state_arrays(g, p + "g_", out)
        state_arrays(d, p + "d_", out)
    hp.discriminator_linguistic_condition = True


def _run_ref_step(ref, tr, hp, g, d, og, od, x, y, lens, R, w_d, mse_w, mge_w, adv_w=1.0):
    """One mini-batch through the reference's own apply_generator / update_discriminator /
    update_generator (train.py:336-355, 245-279, 282-320) exactly as train_loop calls them."""
    lengths = torch.LongTensor(lens)
    y_static = ref.multistream.get_static_features(y, len(hp.windows), hp.stream_sizes, hp.has_dynamic_features)
    mask = ref.seqloss.sequence_mask(lengths).unsqueeze(-1)
    og.zero_grad()
    if od is not None:
        od.zero_grad()
    y_hat, y_hat_static = tr.apply_generator(g, x, R, lens)
    res = {}
    if w_d > 0:
        ld, lf, lr_, rc, fc = tr.update_discriminator(d, od, x, y_static, y_hat_static, lens, mask, "train")
        res.update(loss_d=ld, loss_fake_d=lf, loss_real_d=lr_, real_correct=rc, fake_correct=fc)
    lmse, lmge, ladv, lg = tr.update_generator(g, d, og, x, y, y_hat, y_static, y_hat_static,
                                                adv_w if w_d > 0 else 0.0, lens, mask, "train", mse_w=mse_w,
                                                mge_w=mge_w)
    res.update(loss_mse=lmse, loss_mge=lmge, loss_adv=ladv, loss_g=lg)
    return res, y_hat, y_hat_static


LOSS_KEYS = ("loss_d", "loss_fake_d", "loss_real_d", "loss_mse", "loss_mge", "loss_adv", "loss_g",
             "real_correct", "fake_correct")


def gen_step_models(ref, out):
    """GAN steps of the reference with its non-MLP generators (BASELINE cfg1 / cfg3 / cfg5 at toy sizes,
    dropout 0 so train mode is deterministic): In2OutHighwayNet without a discriminator (w_d = 0),
    In2OutRNNHighwayNet (bidirectional LSTM) + MLP D on hparams.vc, LSTMRNN (bidirectional) + MLP D on
    hparams.tts_acoustic; two consecutive mini-batches each, ragged lengths."""
    tr, hparams, M = ref.train, ref.hparams, ref.models
    from oracle.nnmnkwii_port import unit_variance_mlpg_matrix
    rng = np.random.default_rng(9)
    cases = [
        ("hw_", hparams.vc, lambda: M.In2OutHighwayNet(in_dim=27, out_dim=27, static_dim=9, num_hidden=2,
                                                         hidden_dim=24, dropout=0.0), None, 27, 27, 0.0, 1.0, 1.0),
        ("rhw_", hparams.vc, lambda: M.In2OutRNNHighwayNet(in_dim=27, out_dim=27, static_dim=9, num_hidden=2,
                                                            hidden_dim=12, bidirectional=True, dropout=0.0),
         lambda: M.MLP(in_dim=9, out_dim=1, num_hidden=2, hidden_dim=16, dropout=0.0, last_sigmoid=True),
         27, 27, 1.0, 0.0, 1.0),
        ("lstm_", hparams.tts_acoustic, lambda: M.LSTMRNN(in_dim=20, out_dim=187, num_hidden=2, hidden_dim=16,
                                                          bidirectional=True, dropout=0.0, last_sigmoid=False),
         lambda: M.MLP(in_dim=58, out_dim=1, num_hidden=3, hidden_dim=16, dropout=0.0, last_sigmoid=True),
         20, 187, 1.0, 0.5, 1.0),
    ]
    B, T = 3, 24
    for tag, hp, mk_g, mk_d, d_in, d_out, w_d, mse_w, mge_w in cases:
        saved = (hp.stream_sizes, hp.discriminator_linguistic_condition)
        if hp is hparams.vc:
            hp.stream_sizes = [27]                    # 9 static dims x 3 windows (hparams.py:27 with order 9)
        hp.discriminator_linguistic_condition = False
        tr.hp = hp
        torch.manual_seed(31)
        g = mk_g()
        d = mk_d() if mk_d is not None else None
        g.train()
        state_arrays(g, tag + "g0_", out)
        og = optim.Adagrad(g.parameters(), lr=0.01, weight_decay=1e-7)
        od = None
        if d is not None:
            d.train()
            state_arrays(d, tag + "d0_", out)
            od = optim.Adagrad(d.parameters(), lr=0.01, weight_decay=1e-7)
        R = torch.from_numpy(unit_variance_mlpg_matrix(hp.windows, T))
        for it in range(2):
            lens = lengths_desc(rng, B, T)
            x = torch.randn(B, T, d_in) if hp is hparams.vc else torch.rand(B, T, d_in) * 0.98 + 0.01
            y = torch.randn(B, T, d_out)
            for b, n in enumerate(lens):
                x[b, n:] = 0
                y[b, n:] = 0
            res, y_hat, y_hat_static = _run_ref_step(ref, tr, hp, g, d, og, od, x, y, lens, R, w_d, mse_w, mge_w)
            p = "%sit%d_" % (tag, it)
            out[p + "x"], out[p + "y"], out[p + "lengths"] = npy(x), npy(y), np.array(lens)
            out[p + "y_hat"], out[p + "y_hat_static"] = npy(y_hat), npy(y_hat_static)
            out[p + "losses"] = np.array([res.get(k, np.nan) for k in LOSS_KEYS], dtype=np.float64)
            state_arrays(g, p + "g_", out)
            if d is not None:
                state_arrays(d, p + "d_", out)
        out[tag + "cfg"] = np.array([w_d, mse_w, mge_w], dtype=np.float64)
        hp.stream_sizes, hp.discriminator_linguistic_condition = saved


def gen_eval(ref, out):
    """reference evaluation_tts.py:50-97 ``gen_parameters`` (the call site of nnmnkwii.paramgen.mlpg with unit and
    with real variances), executed UNMODIFIED where it lies: only that function definition is compiled out of the file
    (the module imports pyworld / pysptk / hts question sets at load time), with ``paramgen`` / ``P`` bound to the
    oracle's restatements and ``hp_acoustic`` to the reference's own hparams.tts_acoustic."""
    import ast
    import types
    path = os.path.join(reference_loader.REFERENCE_ROOT, "evaluation_tts.py")
    tree = ast.parse(open(path).read(), path)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "gen_parameters"]
    assert len(fn) == 1
    ns = {"np": np, "paramgen": types.SimpleNamespace(mlpg=nnp.mlpg),
          "P": types.SimpleNamespace(inv_scale=lambda x, m, s: s * x + m), "hp_acoustic": ref.hparams.tts_acoustic}
    exec(compile(ast.Module(body=fn, type_ignores=[]), path, "exec"), ns)
    rng = np.random.RandomState(11)
    T = 90
    y = rng.randn(T, 187)
    mean = {"acoustic": rng.randn(187) * 0.3}
    std = {"acoustic": 0.4 + rng.rand(187)}
    out["eval_y"], out["eval_mean"], out["eval_std"] = y, mean["acoustic"], std["acoustic"]
    for tag, mge in (("mge", True), ("var", False)):
        # the non-MGE branch inv_scales with the dicts themselves at reference evaluation_tts.py:82 (a latent bug of the
        # script: P.inv_scale(y, Y_mean, Y_std) on dict arguments); it is fed the acoustic arrays through a dict-like
        # that also answers ["acoustic"], which is what the following lines index
        if mge:
            mgc, lf0, vuv, bap = ns["gen_parameters"](y.copy(), mean, std, True)
        else:
            class Both(np.ndarray):
                def __getitem__(self, k):
                    return np.asarray(self) if isinstance(k, str) else np.ndarray.__getitem__(self, k)
            mgc, lf0, vuv, bap = ns["gen_parameters"](y.copy(), mean["acoustic"].view(Both), std["acoustic"].view(Both), False)
        for k, v in (("mgc", mgc), ("lf0", lf0), ("vuv", vuv), ("bap", bap)):
            out["eval_%s_%s" % (tag, k)] = np.asarray(v, dtype=np.float64)


def run_reference_unit_tests(ref):
    """Execute the reference's own tests/test_gantts.py (5 tests) where it lies, on top of the nnmnkwii restatement."""
    import importlib.util
    import types
    stubs = reference_loader._stub_modules()
    names = list(stubs) + ["gantts", "gantts.models", "gantts.seqloss", "gantts.multistream"]
    saved = {k: sys.modules.get(k) for k in names}
    try:
        sys.modules.update(stubs)
        pkg = types.ModuleType("gantts")
        pkg.models, pkg.seqloss, pkg.multistream = ref.models, ref.seqloss, ref.multistream
        sys.modules.update({"gantts": pkg, "gantts.models": ref.models,
                            "gantts.seqloss": ref.seqloss, "gantts.multistream": ref.multistream})
        path = os.path.join(reference_loader.REFERENCE_ROOT, "tests", "test_gantts.py")
        spec = importlib.util.spec_from_file_location("_ref_test_gantts", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        ran = 0
        for name in sorted(dir(mod)):
            if name.startswith("test_"):
                getattr(mod, name)()
                ran += 1
        assert ran == 5
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def gen_selftests(ref, out):
    """What the reference computes on the inputs of tests/test_reference_selftests.py (the configurations of the
    reference's tests/test_gantts.py), after checking that those 5 reference tests pass."""
    sys.path.insert(0, os.path.dirname(HERE))
    import test_reference_selftests as st
    run_reference_unit_tests(ref)
    ms = ref.multistream
    sd, x1, xb, yb, lengths = st.model_case()
    model = ref.models.In2OutHighwayNet()
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model.eval()
    R = torch.from_numpy(nnp.unit_variance_mlpg_matrix(WINDOWS[:2], 100))
    out["model_y_static"] = npy(model(torch.from_numpy(x1), R)[1])
    x = torch.from_numpy(xb).requires_grad_(True)
    _, y_hat = model(x, R)
    loss = ref.seqloss.MaskedMSELoss()(y_hat, torch.from_numpy(yb), torch.from_numpy(lengths))
    loss.backward()
    out["model_loss"], out["model_grad_x"] = npy(loss), npy(x.grad)
    a = torch.arange(0, 63).expand(2, 3, 63)
    for code in st.SELECT_CASES:
        out["select_" + code] = npy(ms.select_streams(a, [60, 1, 1, 1], st.streams(code)))
    out["static_stream_sizes"] = ms.get_static_stream_sizes(st.STREAM_SIZES, st.HAS_DYNAMIC, 3)
    s = torch.from_numpy(st.static_input())
    for code in st.STATIC_CASES:
        out["static_" + code] = npy(ms.get_static_features(s, 3, st.STREAM_SIZES, st.HAS_DYNAMIC,
                                                           streams=st.streams(code)))
    R = torch.from_numpy(nnp.unit_variance_mlpg_matrix(WINDOWS, 100))
    out["mlpg_y"] = npy(ms.multi_stream_mlpg(torch.from_numpy(st.multistream_input()), R, st.STREAM_SIZES,
                                             st.HAS_DYNAMIC))


def gen_trainpy_imports():
    """The module-level imports of the reference's train.py and hparams.py, and the model class names hparams.py
    configures (what train.py:773-781 looks up in gantts.models): names only, read with ast."""
    import ast
    imports = []
    for fname in ("train.py", "hparams.py"):
        path = os.path.join(reference_loader.REFERENCE_ROOT, fname)
        for node in ast.parse(open(path).read(), path).body:
            if isinstance(node, ast.Import):
                imports += [{"file": fname, "module": a.name, "names": []} for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                imports.append({"file": fname, "module": node.module, "names": [a.name for a in node.names]})
    ref = reference_loader.load()
    models = {cfg: {k: getattr(ref.hparams, cfg).values()[k] for k in ("generator", "discriminator")}
              for cfg in ("vc", "tts_duration", "tts_acoustic")}
    return {"imports": imports, "models": models}


def main():
    ref = reference_loader.load()
    torch.manual_seed(1234)
    torch.set_num_threads(1)
    if "--only-reference-tests" in sys.argv:
        f = {}
        gen_selftests(ref, f)
        np.savez_compressed(os.path.join(HERE, "selftests.npz"), **f)
        with open(os.path.join(HERE, "trainpy_imports.json"), "w") as fh:
            json.dump(gen_trainpy_imports(), fh, indent=1)
        print("selftests", os.path.getsize(os.path.join(HERE, "selftests.npz")))
        return
    if "--only-eval" in sys.argv:
        e = {}
        gen_eval(ref, e)
        np.savez_compressed(os.path.join(HERE, "eval.npz"), **e)
        print("eval", os.path.getsize(os.path.join(HERE, "eval.npz")))
        return
    if "--only-step-models" in sys.argv:
        d = {}
        gen_step_models(ref, d)
        np.savez_compressed(os.path.join(HERE, "step_models.npz"), **d)
        print("step_models", os.path.getsize(os.path.join(HERE, "step_models.npz")))
        return
    a, b, c = {}, {}, {}
    gen_seqloss(ref, a)
    gen_multistream(ref, a)
    gen_models(ref, b)
    gen_step(ref, c, False, "u_")
    gen_step(ref, c, True, "c_")
    np.savez_compressed(os.path.join(HERE, "ops.npz"), **a)
    np.savez_compressed(os.path.join(HERE, "models.npz"), **b)
    np.savez_compressed(os.path.join(HERE, "step.npz"), **c)
    d = {}
    gen_step_models(ref, d)
    np.savez_compressed(os.path.join(HERE, "step_models.npz"), **d)
    e = {}
    gen_eval(ref, e)
    np.savez_compressed(os.path.join(HERE, "eval.npz"), **e)
    f = {}
    gen_selftests(ref, f)
    np.savez_compressed(os.path.join(HERE, "selftests.npz"), **f)
    with open(os.path.join(HERE, "trainpy_imports.json"), "w") as fh:
        json.dump(gen_trainpy_imports(), fh, indent=1)
    for n in ("ops", "models", "step", "step_models", "eval", "selftests"):
        print(n, os.path.getsize(os.path.join(HERE, n + ".npz")))


if __name__ == "__main__":
    main()
