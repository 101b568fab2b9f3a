"""bench.py -- GAN-step frames/sec of the B200 hot path (BASELINE.json metric) + roofline + CPU baseline.

    python bench.py --gpus N --steps K --warmup W               # our arm (N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K ...      # the reference's CPU path (pinned oracle port)
    python bench.py --workload cfg3|cfg5 ...                     # the recurrent-generator configurations

A "step" is one full GAN training step (reference train.py:538-580: zero_grad, generator forward, MLPG,
discriminator update, generator update, both clip+Adagrad steps) over one synthetic batch.  Default workload =
cfg2, the configuration BASELINE.json quotes the metric on: TTS acoustic MLP generator (425-512-512-512-187) + MLP
discriminator on the 58 masked mgc dims (58-256-256-256-1), B=32 x T=1000 padded frames PER GPU (weak scaling),
dropout 0.5 in train mode, full-length utterances.  cfg3 = VC In2OutRNNHighwayNet (3 x 512 BiLSTM) + MLP D, B=16 x
T=2000; cfg5 = TTS LSTMRNN (3 x 512 BiLSTM) + MLP D + MGE, B=64 x T=1500 per GPU.

Timing: W untimed warm-up steps, then exactly K steps are timed with CUDA events between barriers (pick K so that
the window lasts a second or more: a 20-step window of a 1.3 ms step is 0.03 s and measures mostly noise).

--dump-outputs DIR: after the timed steps, what the last of them computed -- the losses, y_hat and y_hat_static the
step hands its caller and the generator and discriminator parameters it updated -- is written as DIR/<name>.npy
(float32; a fixed seeded sample of the elements where the whole would exceed 64 MB).  Inputs and initial weights are
seeded, so two builds run with the same arguments can be compared output for output.

One JSON line on stdout (rank 0).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True       # the tree may be read-only; the benchmark writes nothing into it
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "compat"))

WINDOWS = [(0, 0, np.array([1.0])), (1, 1, np.array([-0.5, 0.0, 0.5])), (1, 1, np.array([1.0, -2.0, 1.0]))]
TTS_HP = dict(stream_sizes=[180, 3, 1, 3], has_dynamic_features=[True, True, False, True],
              adversarial_streams=[True, False, False, False], mask_nth_mgc_for_adv_loss=2, num_windows=3,
              discriminator_linguistic_condition=False)
VC_HP = dict(stream_sizes=[177], has_dynamic_features=[True], adversarial_streams=[True], mask_nth_mgc_for_adv_loss=0,
             num_windows=3, discriminator_linguistic_condition=False)

WORKLOADS = {
    "cfg2": dict(kind="mlp", B=32, T=1000, d_in=425, d_out=187, g_hidden=512, g_layers=3, d_dims=[58, 256, 256, 256, 1],
                 dropout_g=0.5, dropout_d=0.5, hp=TTS_HP, uniform_x=True,
                 text="cfg2: TTS acoustic MLP G 425-512-512-512-187 + MLP D 58-256-256-256-1 (mgc adv, mask_nth=2), "
                      "B=32 T=1000 per GPU, MGE(MLPG)+ADV, dropout 0.5, Adagrad"),
    "cfg3": dict(kind="rnn_highway", B=16, T=2000, d_in=177, d_out=177, static_dim=59, g_hidden=512, g_layers=3,
                 d_dims=[59, 256, 256, 1], dropout_g=0.5, dropout_d=0.5, hp=VC_HP, uniform_x=False,
                 text="cfg3: VC In2OutRNNHighwayNet 177->177 (static 59, 3 x 512 bidirectional LSTM, dropout 0.5) + MLP D "
                      "59-256-256-1, B=16 T=2000 per GPU, MGE(MLPG)+ADV, Adagrad"),
    "cfg5": dict(kind="lstm", B=64, T=1500, d_in=425, d_out=187, g_hidden=512, g_layers=3, d_dims=[58, 256, 256, 256, 1],
                 dropout_g=0.0, dropout_d=0.5, hp=TTS_HP, uniform_x=True,
                 text="cfg5: TTS acoustic LSTMRNN 425->187 (3 x 512 bidirectional) + MLP D 58-256-256-256-1 (mgc adv, "
                      "mask_nth=2), B=64 T=1500 per GPU, MGE(MLPG)+ADV, Adagrad"),
}
NUM_BATCHES = 4          # ring of distinct synthetic batches (larger than the 126 MB L2 for every workload)
DUMP_BYTES = 64 << 20    # --dump-outputs: at most this much in all
NPY_HEADER_BYTES = 128


def algorithmic_flops_per_frame(w):
    """SURVEY.md 8d, de-duplicated GAN step (1 MAC = 2 FLOP): generator fwd + one bwd (no input gradient), three
    discriminator forwards, D bwd real (no input gradient) + fake, adv-D bwd (input gradient only):
    MAC/frame = 3 F_G - k0 + 8 F_D - d_h1 d_in."""
    dd = w["d_dims"]
    F_D = sum(a * b for a, b in zip(dd[:-1], dd[1:]))
    d_part = 8 * F_D - dd[1] * dd[0]
    if w["kind"] == "mlp":
        g_dims = [w["d_in"]] + [w["g_hidden"]] * w["g_layers"] + [w["d_out"]]
        F_G = sum(a * b for a, b in zip(g_dims[:-1], g_dims[1:]))
        return 2.0 * (3 * F_G - g_dims[0] * g_dims[1] + d_part)
    H, dirs = w["g_hidden"], 2
    F_L, inp = 0, w["d_in"]
    for _ in range(w["g_layers"]):
        F_L += dirs * 4 * H * (inp + H)
        inp = dirs * H
    F_O = dirs * H * w["d_out"]
    gate = w.get("static_dim", 0) ** 2
    return 2.0 * (3 * (F_L + F_O) - dirs * 4 * H * w["d_in"] + 2 * gate + d_part)


def make_batches(w, seed, n, pinned, B=None):
    g = torch.Generator().manual_seed(seed)
    B = B or w["B"]
    out = []
    for _ in range(n):
        if w["uniform_x"]:
            x = torch.rand(B, w["T"], w["d_in"], generator=g) * 0.98 + 0.01
        else:
            x = torch.randn(B, w["T"], w["d_in"], generator=g)
        y = torch.randn(B, w["T"], w["d_out"], generator=g)
        if pinned:
            x, y = x.pin_memory(), y.pin_memory()
        out.append((x, y))
    return out


def dump_outputs(arrays, out_dir, budget=DUMP_BYTES):
    """Write {name: float32/float64 array} as out_dir/<name>.npy, at most `budget` bytes in all.  Smallest first, each
    array gets an equal share of what is left; one that does not fit is replaced by a sample of its flattened
    elements, drawn with a fixed seed and kept in index order, so runs with the same shapes sample the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: (kv[1].nbytes, kv[0]))
    left = budget
    for i, (name, a) in enumerate(items):
        share = left // (len(items) - i) - NPY_HEADER_BYTES
        if a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes + NPY_HEADER_BYTES


class ClockSampler(object):
    """SM clock / throttle reasons sampled DURING the timed region (NVML polling thread; falls back to an
    `nvidia-smi -lms 100` subprocess when the NVML bindings are unavailable)."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml = index, [], None, None
        self.sm, self.mask, self.max_mhz, self._stop = [], 0, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            props = torch.cuda.get_device_properties(self.index)
            bus = props.pci_bus_id if hasattr(props, "pci_bus_id") else None
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index) if bus is None else None
            if self.handle is None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.handle = h
                        break
                if self.handle is None:
                    self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self._stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            reasons = sorted(v for k, v in self.REASONS.items() if self.mask & k)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": reasons, "samples": len(self.sm), "how": "NVML poll every 5 ms"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "how": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------ CPU baseline
def cpu_reference_step_runner(w, sample_B, threads):
    """The reference's CPU path (pinned oracle port of gantts/*.py + train.py step functions, torch CPU fp32,
    dense-R MLPG exactly like the reference) on `sample_B` utterances of the workload's T and widths.  Returns a
    closure running one step, the frames it processes and the seconds the dense R construction took."""
    from oracle import gantts_port as gp
    from oracle import nnmnkwii_port as nnp
    torch.set_num_threads(threads)
    torch.manual_seed(1234)
    lin = lambda i, o: torch.nn.Linear(i, o)
    dd = w["d_dims"]
    d_layers = [(l.weight.detach().clone().requires_grad_(True), l.bias.detach().clone().requires_grad_(True))
                for l in (lin(a, b) for a, b in zip(dd[:-1], dd[1:]))]
    d_sum = [torch.zeros_like(t) for pair in d_layers for t in pair]
    hp = w["hp"]
    (x, y), = make_batches(w, 1234, 1, False, B=sample_B)
    lens = [w["T"]] * sample_B
    t0 = time.perf_counter()
    R = torch.from_numpy(nnp.unit_variance_mlpg_matrix(WINDOWS, w["T"]))    # train.py:510-513, rebuilt per batch there
    r_seconds = time.perf_counter() - t0
    if w["kind"] == "mlp":
        g_dims = [w["d_in"]] + [w["g_hidden"]] * w["g_layers"] + [w["d_out"]]
        mods = [lin(a, b) for a, b in zip(g_dims[:-1], g_dims[1:])]
        sd = {}
        for i, m in enumerate(mods[:-1]):
            sd["layers.%d.weight" % i], sd["layers.%d.bias" % i] = m.weight.detach().numpy(), m.bias.detach().numpy()
        sd["last_linear.weight"], sd["last_linear.bias"] = mods[-1].weight.detach().numpy(), mods[-1].bias.detach().numpy()
        gen = gp.GeneratorOracle("mlp", sd)
    else:
        lstm = torch.nn.LSTM(w["d_in"], w["g_hidden"], w["g_layers"], batch_first=True, bidirectional=True)
        h2o = lin(2 * w["g_hidden"], w["d_out"])
        sd = {"lstm." + k: v.detach().numpy() for k, v in lstm.state_dict().items()}
        sd["hidden2out.weight"], sd["hidden2out.bias"] = h2o.weight.detach().numpy(), h2o.bias.detach().numpy()
        kw = dict(num_hidden=w["g_layers"], hidden_dim=w["g_hidden"], bidirectional=True)
        if w["kind"] == "rnn_highway":
            gate = lin(w["static_dim"], w["static_dim"])
            sd["T.weight"], sd["T.bias"] = gate.weight.detach().numpy(), gate.bias.detach().numpy()
            gen = gp.GeneratorOracle("rnn_highway", sd, static_dim=w["static_dim"], **kw)
        else:
            gen = gp.GeneratorOracle("lstm", sd, **kw)

    def run():
        gp.gan_step(lambda: gen.forward(x, R, lens, hp, w["dropout_g"], True), gen.params(), gen.sums, d_layers, d_sum,
                    x, y, lens, R, hp, w_d=1.0, mse_w=0.0, mge_w=1.0, adv_w=1.0, dropout_d=w["dropout_d"], training=True)
    return run, sample_B * w["T"], r_seconds


def time_cpu_baseline(w, steps, warmup, full_batch, time_budget_s=None):
    """Reference CPU arm.  torch's CPU kernels do not scale to every core of a large host on these shapes (128
    threads were 3x slower than 32 on the B200 box), so a one-step probe picks the fastest thread count among
    {16, 32, 64, all}.  `full_batch`: time the whole B-utterance batch (same config as the GPU arm); when one step of
    it takes longer than 30 s -- or for the default in-line baseline of the GPU arm -- a bounded sample of utterances
    is timed instead (frames/s is per padded frame, so the sample measures the same quantity)."""
    ncpu = os.cpu_count() or 1
    cands = sorted(set(min(c, ncpu) for c in (16, 32, 64, ncpu)))
    small = 2 if w["kind"] != "mlp" else 4
    sample_B = w["B"] if full_batch else small
    run, frames, r_s = cpu_reference_step_runner(w, sample_B, cands[0])
    t0 = time.perf_counter()
    run()                                   # first-touch / allocator warm-up
    first = time.perf_counter() - t0
    if full_batch and first > 30.0:
        sample_B = small
        run, frames, r_s = cpu_reference_step_runner(w, sample_B, cands[0])
        run()
    best, best_dt = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best, best_dt = c, dt
    torch.set_num_threads(best)
    if time_budget_s is not None:
        # the reference arm honours --steps / --warmup as far as the time budget allows (CPU steps take seconds each)
        steps = max(2, min(steps, int(time_budget_s / max(best_dt, 1e-3))))
        warmup = max(1, min(warmup, int(0.25 * time_budget_s / max(best_dt, 1e-3))))
    for _ in range(max(0, warmup - 1)):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    return {"value": frames / dt, "unit": "frames/s", "cores": best, "kind": "port",
            "sample": "%d of %d utterances x T=%d per step, %d timed steps, dense-R MLPG with R prebuilt (building R "
                      "for T=%d takes %.2f s on this host; train.py:510-513 rebuilds it every batch: %.0f frames/s "
                      "with that included), torch %s CPU fp32, thread count picked from %s of %d host cores by a "
                      "one-step probe" % (sample_B, w["B"], w["T"], steps, w["T"], r_s, frames / (dt + r_s),
                                          torch.__version__, cands, ncpu),
            "ms_per_step": dt * 1e3, "same_config_as_gpu_arm": sample_B == w["B"],
            "value_with_R_build": frames / (dt + r_s), "steps_timed": steps, "warmup_run": warmup}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    cb = time_cpu_baseline(w, max(2, args.steps), max(1, args.warmup), full_batch=True, time_budget_s=90.0)
    steps, warmup = cb["steps_timed"], cb["warmup_run"]
    line = {"impl": "reference", "metric": "gan_step_frames_per_sec", "value": cb["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, "cpu", args), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU steps take seconds each: the arm runs --steps/--warmup as far as a 90 s budget of timed work allows "
                    "(here %d timed steps after %d warm-up) so that the run ends within minutes" % (steps, warmup)}
    emit_json_line(line)


def workload_config(w, engine, args=None):
    bytes_per_batch = w["B"] * w["T"] * (w["d_in"] + w["d_out"]) * 4
    return {"workload": w["text"], "global_batch_per_gpu": w["B"], "seq_len": w["T"], "engine": engine,
            "l2": "per-step working set > 1 GB and a ring of %d distinct input batches (%d MB) exceed the 126 MB L2; "
                  "no explicit flush" % (NUM_BATCHES, NUM_BATCHES * bytes_per_batch // (1 << 20)),
            "timing": "one window of exactly K = --steps steps, CUDA events, barrier + synchronize on both sides, "
                      "max over ranks",
            "parallelism": "utterance-sharded data parallel, one NCCL SUM all-reduce per model per step"}


_REAL_STDOUT_FD = None


def redirect_stdout_to_stderr():
    global _REAL_STDOUT_FD
    if _REAL_STDOUT_FD is None:
        sys.stdout.flush()
        _REAL_STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(line):
    text = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT_FD is None:
        os.write(1, text)
    else:
        os.write(_REAL_STDOUT_FD, text)


# ------------------------------------------------------------------------------------ B200 arm
def build_models(w, dev):
    import gantts_b200
    M = gantts_b200.models
    dd = w["d_dims"]
    md = M.MLP(dd[0], 1, len(dd) - 2, dd[1], dropout=w["dropout_d"], last_sigmoid=True)
    if w["kind"] == "mlp":
        mg = M.MLP(w["d_in"], w["d_out"], w["g_layers"], w["g_hidden"], dropout=w["dropout_g"], last_sigmoid=False)
    elif w["kind"] == "rnn_highway":
        mg = M.In2OutRNNHighwayNet(in_dim=w["d_in"], out_dim=w["d_out"], static_dim=w["static_dim"],
                                   num_hidden=w["g_layers"], hidden_dim=w["g_hidden"], bidirectional=True,
                                   dropout=w["dropout_g"])
    else:
        mg = M.LSTMRNN(in_dim=w["d_in"], out_dim=w["d_out"], num_hidden=w["g_layers"], hidden_dim=w["g_hidden"],
                       bidirectional=True, dropout=w["dropout_g"], last_sigmoid=False)
    return mg.to(dev).train(), md.to(dev).train()


def run_b200_arm(args):
    if os.environ.get("GANTTS_B200_DBG", "0") not in ("", "0") or os.environ.get("GANTTS_B200_CHAIN_DBG", "0") not in ("", "0"):
        raise SystemExit("bench.py: GANTTS_B200_DBG is a phase-timing switch that skips work inside the kernels; "
                         "refusing to produce a benchmark line with it set")
    from gantts_b200 import parallel
    # stdout carries exactly ONE JSON line.  NCCL prints its version banner with a bare printf on fd 1 during
    # the first communicator init (NCCL_DEBUG_FILE does not catch it), so fd 1 points at stderr for the whole
    # run and the JSON line is written to the saved descriptor (emit_json_line).
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    redirect_stdout_to_stderr()
    rank, world, local = parallel.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # the library comes from `python -m gantts_b200.build` (or __graft_entry__.build()); the benchmark only loads
    # it, so it runs from a read-only tree
    import gantts_b200
    from gantts_b200 import _lib, step as gstep, config
    from nnmnkwii.paramgen import unit_variance_mlpg_matrix   # compat shim (product side, memoised)
    lib = _lib.load()
    config.engine = args.engine
    w = WORKLOADS[args.workload]
    fused_ok = w["kind"] == "mlp"
    path = args.path if fused_ok else "modular"
    torch.manual_seed(1234)
    mg, md = build_models(w, dev)
    hpd = w["hp"]
    hp = gstep.HParams(windows=WINDOWS, stream_sizes=hpd["stream_sizes"], has_dynamic_features=hpd["has_dynamic_features"],
                       adversarial_streams=hpd["adversarial_streams"],
                       mask_nth_mgc_for_adv_loss=hpd["mask_nth_mgc_for_adv_loss"],
                       discriminator_linguistic_condition=False)
    lengths = torch.full((w["B"],), w["T"], dtype=torch.int64, device=dev)
    frames_per_step = w["B"] * w["T"] * world

    class Runner(object):
        """path 'fused': gantts_gan_step (one C call per mini-batch); 'modular': GanTrainer."""

        def __init__(self):
            if path == "fused":
                from gantts_b200 import fused
                self.fs = fused.FusedGanStep(mg, md, hp, w["B"], w["T"], w_d=1.0, mse_w=0.0, mge_w=1.0)
            else:
                self.tr = gstep.GanTrainer(mg, md, hp, w_d=1.0, mse_w=0.0, mge_w=1.0)
                self.R = torch.from_numpy(unit_variance_mlpg_matrix(hp.windows, w["T"])).to(dev)

        def step(self, x, y):
            if path == "fused":
                losses = self.fs.step(x, y, lengths, frames=frames_per_step)
                return {"loss_d": losses[0], "loss_mge": losses[4], "loss_adv": losses[5], "loss_g": losses[6]}
            self.last = self.tr.step(x, y, lengths, self.R)
            return self.last[0]

        def outputs(self):
            """What the last step handed its caller, and the parameters it updated: {name: float32 array}."""
            if path == "fused":
                from gantts_b200.fused import LOSS_NAMES
                out = dict(zip(LOSS_NAMES, self.fs.losses.detach().cpu().unbind()))
                out["y_hat"], out["y_hat_static"] = self.fs.y_hat, self.fs.y_hat_static
            else:
                out = dict(self.last[0])
                out["y_hat"], out["y_hat_static"] = self.last[1], self.last[2]
            for tag, m in (("g", mg), ("d", md)):
                out.update(("%s.%s" % (tag, k), p) for k, p in m.named_parameters())
            return {k: torch.as_tensor(v).detach().float().cpu().numpy() for k, v in out.items()}

        def nccl_warmup(self):
            if world == 1:
                return
            bufs = [self.fs.grad_buffer(0), self.fs.grad_buffer(1)] if path == "fused" else \
                [self.tr.opt_g.flat_grad, self.tr.opt_d.flat_grad]
            for _ in range(12):                      # NCCL sets its channels up lazily per message size
                for b in bufs:
                    parallel.allreduce_sum_(b)
            for b in bufs:
                b.zero_()

    trainer = Runner()
    host = make_batches(w, 1234 + rank, NUM_BATCHES, pinned=True)
    resident = [(x.to(dev), y.to(dev)) for x, y in host]

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(loop):
        """loop(K) enqueues K = --steps steps; returns ms per step over that one window (max over ranks)."""
        barrier()
        t_host = time.perf_counter()
        e0.record()
        loop(args.steps)
        e1.record()
        t_host = time.perf_counter() - t_host
        barrier()
        local_ms = e0.elapsed_time(e1)
        ms = max_over_ranks(local_ms)
        if os.environ.get("GANTTS_B200_BENCH_TRACE"):
            sys.stderr.write("[trace] rank %d: device %.3f ms/step (max over ranks %.3f), host enqueue %.3f ms/step\n"
                             % (rank, local_ms / args.steps, ms / args.steps, t_host / args.steps * 1e3))
            sys.stderr.flush()
        return ms / args.steps

    # ---------------- value: inputs resident in HBM
    trainer.nccl_warmup()
    for i in range(args.warmup):
        trainer.step(*resident[i % NUM_BATCHES])
    barrier()
    if os.environ.get("GANTTS_B200_CUDA_PROFILE_STEPS"):
        # profiler window (ncu --profile-from-start off): exactly N steps after the warm-up, so that a launch list or
        # a --set full capture holds whole steps in launch order.  Numbers printed by such a run are never bench values.
        torch.cuda.profiler.start()
        for i in range(int(os.environ["GANTTS_B200_CUDA_PROFILE_STEPS"])):
            trainer.step(*resident[i % NUM_BATCHES])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last = {}

    def resident_loop(n):
        for i in range(n):
            last["out"] = trainer.step(*resident[i % NUM_BATCHES])

    launches0 = lib.gantts_launch_count()
    ms_per_step = timed(resident_loop)
    launches = (lib.gantts_launch_count() - launches0) / float(args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(trainer.outputs(), args.dump_outputs)
    value = frames_per_step / (ms_per_step * 1e-3)
    loss_g = float(last["out"]["loss_g"])
    # host time to ENQUEUE a step (8 steps stay well inside the driver's launch queue, so the CPU never waits for the
    # GPU): while it is below ms_per_step the GPU is never starved and a CUDA graph of the step would not change `value`
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    resident_loop(8)
    host_enqueue_ms = (time.perf_counter() - t0) / 8 * 1e3
    torch.cuda.synchronize()
    # ---------------- roofline pass: K steps again with CUDA events around every GEMM / chain / MLPG / LSTM launch
    # (kept out of the region `value` is timed on: the event records sit between consecutive kernels)
    lib.gantts_profile_enable(1)
    resident_loop(args.steps)
    torch.cuda.synchronize()
    lib.gantts_profile_enable(0)
    pms, pwork, pn = (ctypes.c_double * 8)(), (ctypes.c_double * 8)(), (ctypes.c_longlong * 8)()
    _lib.check(lib.gantts_profile_collect(pms, pwork, pn))

    # ---------------- e2e: host buffers in, losses out, copies inside the timed region
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(resident[0][0]), torch.empty_like(resident[0][1])) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.empty(4, dtype=torch.float32).pin_memory()

    def prefetch(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            bufs[slot][0].copy_(host[i % NUM_BATCHES][0], non_blocking=True)
            bufs[slot][1].copy_(host[i % NUM_BATCHES][1], non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_loop(n):
        prefetch(0)
        for i in range(n):
            if i + 1 < n:
                prefetch(i + 1)
            slot = i % 2
            torch.cuda.current_stream().wait_event(ready[slot])
            o = trainer.step(bufs[slot][0], bufs[slot][1])
            consumed[slot].record()
            loss_host.copy_(torch.stack([o["loss_g"], o["loss_d"], o["loss_mge"], o["loss_adv"]]).detach(),
                            non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for ev in consumed:
        ev.record()
    e2e_loop(max(2, min(args.warmup, 4)))
    e2e_ms = timed(e2e_loop)
    h2d = sum(t.numel() * 4 for t in host[0])

    # ---------------- N > 1: what the two gradient all-reduces of a step cost by themselves (back to back, no skew to
    # absorb): the residual the data-parallel step pays over the single-GPU step, reported next to it
    allreduce = None
    if world > 1 and path == "fused":
        gbufs = [trainer.fs.grad_buffer(1).clone(), trainer.fs.grad_buffer(0).clone()]

        def ar_loop(n):
            for _ in range(n):
                for b in gbufs:
                    parallel.allreduce_sum_(b)
                    b.mul_(1.0 / world)             # keeps the values bounded over the repeats

        ar_loop(5)
        ar_ms = timed(ar_loop)
        allreduce = {"us_per_step_pair": ar_ms * 1e3, "d_bytes": gbufs[0].numel() * 4, "g_bytes": gbufs[1].numel() * 4,
                     "note": "D + G gradient all-reduce (NCCL) + one scale kernel each, timed alone"}

    # ---------------- drop-in path (cfg2, one process): the reference's own per-batch logic -- tests/trainpy_mirror.py =
    # train.py:528-580 with its inline BCE, its .item() calls, clip_grad_norm_ and torch.optim.Adagrad -- on the
    # `gantts` alias package (the B200 modules), dense R on the device as train.py builds it
    dropin = None
    if world == 1 and w["kind"] == "mlp" and not args.no_dropin:
        sys.path.insert(1, os.path.join(ROOT, "tests"))
        import trainpy_mirror
        torch.manual_seed(1234)
        g2, d2 = build_models(w, dev)
        og = torch.optim.Adagrad(g2.parameters(), lr=0.01, weight_decay=1e-7)
        od = torch.optim.Adagrad(d2.parameters(), lr=0.01, weight_decay=1e-7)
        Rd = torch.from_numpy(unit_variance_mlpg_matrix(hp.windows, w["T"])).to(dev)
        cpu_lengths = [w["T"]] * w["B"]

        def dropin_loop(n):
            for i in range(n):
                x, y = resident[i % NUM_BATCHES]
                trainpy_mirror.train_step(g2, d2, og, od, x, y, lengths, Rd, hp)
        dropin_loop(3)
        torch.cuda.synchronize()
        l0 = lib.gantts_launch_count()
        n_d = max(10, min(args.steps, 30))
        t0 = time.perf_counter()
        dropin_loop(n_d)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / n_d
        dropin = {"ms_per_step": dt * 1e3, "frames_per_sec": w["B"] * w["T"] / dt,
                  "native_launches_per_step": (lib.gantts_launch_count() - l0) / n_d, "host_syncs_per_step": 10,
                  "vs_fused_step": dt * 1e3 / ms_per_step,
                  "how": "tests/trainpy_mirror.train_step (reference train.py:528-580 re-typed: 10 .item() host "
                         "syncs, torch clip_grad_norm_, torch.optim.Adagrad) on gantts.models.MLP x 2, dense R "
                         "resident on the device; wall clock over %d steps" % n_d}
        del g2, d2, og, od

    if rank != 0:
        return
    # ---------------- roofline of the dominant kernel family
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    kinds = {0: "gemm_bf16x3_kernel<K-major>", 1: "gemm_bf16x3_kernel<MN-major>", 2: "mlpg_fwd_kernel",
             3: "mlpg_bwd_kernel", 4: "lstm_fwd_kernel", 5: "lstm_bwd_kernel", 6: "chain_pair_kernel"}
    per_kind = {}
    for k, name in kinds.items():
        if pn[k]:
            per_kind[name] = {"ms_per_step": pms[k] / args.steps, "launches_per_step": pn[k] / args.steps,
                              "work_per_step": pwork[k] / args.steps,
                              "achieved": (pwork[k] / (pms[k] * 1e-3)) / (1e9 if k in (2, 3) else 1e12),
                              "unit": "GB/s" if k in (2, 3) else "TFLOP/s"}
    tensor_kinds = (0, 1, 6)
    fam_ms = sum(pms[k] for k in tensor_kinds)
    fam_work = sum(pwork[k] for k in tensor_kinds)
    fam_ach = (fam_work / (fam_ms * 1e-3)) / 1e12 if fam_ms else 0.0
    if w["kind"] == "mlp":
        dom = max(tensor_kinds, key=lambda k: pms[k])
    else:
        dom = max((4, 5), key=lambda k: pms[k])
    ach = (pwork[dom] / (pms[dom] * 1e-3)) / 1e12 if pms[dom] else 0.0
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_top_kernel.json")))
        traffic = prof.get("dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"kernel": kinds[dom], "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": ach / peak_tf, "traffic": traffic, "peak_source": peak_src,
                "note": "achieved = algorithmic fp32-equivalent FLOPs (2MNK per GEMM) / CUDA-event time of the "
                        "launches (second pass of the same K steps with an event pair around every launch); the "
                        "bf16x3 split executes 3 tensor-core MMAs per algorithmic product, so executed bf16 pipe "
                        "rate = 3 x achieved" if w["kind"] == "mlp" else
                        "dominant kernel = the LSTM recurrence (one cooperative launch per layer: T sequential steps, "
                        "exact-fp32 FFMA with W_hh in registers): latency-bound, reported against the tensor peak as "
                        "the contract asks; its share of the step is what matters",
                "tensor_pipe_frac_executed": 3.0 * ach / peak_tf if w["kind"] == "mlp" else None,
                "gemm_family": {"ms_per_step": fam_ms / args.steps, "achieved_tflops_algorithmic": fam_ach,
                                "frac_algorithmic": fam_ach / peak_tf, "tensor_pipe_frac_executed": 3.0 * fam_ach / peak_tf,
                                "launches_per_step": sum(pn[k] for k in tensor_kinds) / args.steps},
                "share_of_step": (pms[dom] / args.steps) / ms_per_step,
                "kernels": per_kind}
    cb = None
    if world == 1 and not args.no_cpu_baseline:
        cb = time_cpu_baseline(w, steps=3 if w["kind"] == "mlp" else 2, warmup=1, full_batch=False)
    line = {"metric": "gan_step_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (GEMMs: bf16x3 split on tcgen05, fp32 accumulate)" if args.engine == "tc" else "f32",
            "data": "synthetic", "config": workload_config(w, args.engine, args), "clocks": clocks,
            "e2e": {"value": frames_per_step / (e2e_ms * 1e-3), "unit": "frames/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                    "how": "pinned host x,y -> double-buffered cudaMemcpyAsync on a copy stream -> one step through the "
                           "public API (%s) -> 4 loss scalars D2H; copies inside the timed region" % path},
            "gpu_launches": int(round(launches * args.steps)), "gpu_launches_per_step": launches,
            "host_enqueue_ms_per_step": host_enqueue_ms,
            "algorithmic_gflop_per_step": algorithmic_flops_per_frame(w) * w["B"] * w["T"] / 1e9,
            "step_tflops_algorithmic": algorithmic_flops_per_frame(w) * frames_per_step / (ms_per_step * 1e-3) / 1e12 / world,
            "roofline": roofline, "loss_g_last": loss_g,
            "path": "gantts_gan_step (one C call per mini-batch)" if path == "fused" else "GanTrainer (python-orchestrated native ops)"}
    if allreduce is not None:
        line["allreduce"] = allreduce
    if dropin is not None:
        line["dropin"] = dropin
    if cb is not None:
        line["cpu_baseline"] = cb
    emit_json_line(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--engine", default=os.environ.get("GANTTS_B200_ENGINE", "tc"), choices=["tc", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dropin", action="store_true")
    ap.add_argument("--path", default="fused", choices=["fused", "modular"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
