#!/usr/bin/env python
"""Benchmark of the DCLL hot path: RadioML IQ windows/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one batch of synthetic IQ windows pushed through the whole hot path: IQ->spike encoding
followed by T = 1024 timesteps of radio_ml_conv DCLL training (forward, local loss gradient, weight gradient
and Adam step per layer per timestep), or of inference for the infer workloads.  Prints ONE JSON line.

  value        windows/s with the IQ records already resident in HBM (encode + T timesteps timed)
  e2e          the same through the public API with HOST buffers: pinned-host IQ -> H2D -> iq2spiketrain ->
               ConvNetwork.learn_window -> device vote -> D2H of the per-sample predictions, all timed
  roofline     the kernel class with the largest share of the step (CUDA events sampled inside the timed region on the
               launching stream), plus the other big kernels under roofline.kernels
  precision    default f16x2: tcgen05 tensor cores, fp16 traces against split-fp16 weights / local gradients, two products per
               MAC (DESIGN.md section 6: spike-flip rate <= 1e-3, held-out accuracy within 0.5 pt of FP32 -- both tested)
  fp32_mode    the same workload in the FP32-exact parity mode (BASELINE.json configs[0] says FP32), short run
  bf16x3_mode  the same workload in the three-product split-bf16 tensor-core mode, short run
  other_workloads   the other BASELINE.json configs (mnist_conv, quantised radio_ml_conv_ref, 16x16 script geometry,
               inference sweep points), short runs through the same public API
  cpu_baseline the reference's own classes (oracle/_ref, vendored unmodified by oracle/make_ref.py) on the box's host
               cores, on a bounded sample of the same workload; the oracle port when oracle/_ref is absent

--impl reference times that CPU arm alone, on the same `config`.

--dump-outputs DIR writes what the last timed step handed back to its caller -- the per-timestep class votes, every
layer's parameters and, for training workloads, its neuron state -- as DIR/<name>.npy (float32), so that two builds run
with the same arguments (hence the same seeded inputs) can be compared output for output.  Arrays larger than
DUMP_SAMPLE elements are stored as a fixed seeded sample of DUMP_SAMPLE elements (<name>_sample.npy).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (spec, resolution, per-GPU batch, train, arp, burnin)
    "radio_ml_conv_train_128x128_B64": ("radio_ml_conv", 128, 64, True, 0.0, 50),   # train.py argparse defaults
    "radio_ml_conv_train_16x16_B64": ("radio_ml_conv", 16, 64, True, 0.0, 50),
    "radio_ml_conv_train_16x16_B512_arp": ("radio_ml_conv", 16, 512, True, 1.0, 20),  # scripts/train_radio_ml.sh
    "radio_ml_conv_infer_16x16_B4096": ("radio_ml_conv", 16, 4096, False, 1.0, 20),
    "radio_ml_conv_infer_128x128_B64": ("radio_ml_conv", 128, 64, False, 0.0, 50),
    "radio_ml_conv_train_16x16_B1024": ("radio_ml_conv", 16, 1024, True, 0.0, 50),   # config 5 shard (8192 / 8)
    # BASELINE.json configs[4]: data-parallel training at GLOBAL batch 8192 (per-GPU batch = 8192 / N: strong scaling).
    # 16x16 (script geometry) fits any N; 128x128 needs ~50 GB of state per 1024 samples, i.e. N = 8.
    "radio_ml_conv_train_dp_global8192_16x16": ("radio_ml_conv", 16, -8192, True, 0.0, 50),
    "radio_ml_conv_train_dp_global8192_128x128": ("radio_ml_conv", 128, -8192, True, 0.0, 50),
}
DEFAULT = "radio_ml_conv_train_128x128_B64"
K_CLASSES, N_IQ = 24, 1024
DUMP_SAMPLE = 1 << 20          # elements kept per dumped array (4 MB): under 64 MB for every workload's arrays


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops_sustained"], tensor_burst=d["bf16_tflops"], src="measured")
    return dict(hbm=6650.0, tensor=1400.0, tensor_burst=1590.0, src="fallback")


def flops_per_sample_timestep(res, train):
    # SURVEY.md section 8d: conv fwd 2*Cin*kh*kw*Cout*H'*W' per layer, read-outs 2*F*K (x2 on the last layer)
    hw = res * res
    conv = 2 * 49 * hw * (1 * 32 + 32 * 32 + 32 * 32)
    ro = 2 * (32 * hw) * K_CLASSES * 4
    return (conv + ro) * (2 if train else 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 5]
        os.unlink(self.f.name)
        sm = sorted(int(r[0]) for r in rows if r[0].strip().isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any("Active" == r[2 + i].strip() for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(rows[0][1]) if rows and rows[0][1].strip().isdigit() else None,
                "reasons": reasons, "samples": len(rows)}


def synth(batch, seed):
    """SURVEY section 8d synthetic input: x ~ N(0, 0.4^2) f32 (B,2,1,1024) in the loader layout, uniform labels."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(batch, 2, 1, N_IQ, generator=g) * 0.4).float()
    lab = torch.randint(0, K_CLASSES, (batch,), generator=g)
    y = torch.zeros(batch, K_CLASSES).scatter_(1, lab.unsqueeze(-1), 1)
    return x, y


# --------------------------------------------------------------------------------------------------------
# workload helpers shared by both arms
# --------------------------------------------------------------------------------------------------------
def workload(name, world=1):
    """(spec, resolution, per-GPU batch, train, arp, burnin, scaling).  A negative batch in WORKLOADS is a GLOBAL batch
    split over the ranks (BASELINE.json configs[4]: strong scaling)."""
    spec, res, batch, train, arp, burnin = WORKLOADS[name]
    scaling = "weak"
    if batch < 0:
        if (-batch) % world:
            raise SystemExit("global batch %d does not divide over %d GPUs" % (-batch, world))
        batch, scaling = (-batch) // world, "strong"
    return spec, res, batch, train, arp, burnin, scaling


def config_dict(a, world):
    """`config` of the JSON line -- built by ONE function for both arms so that the driver's same_config check compares
    like with like.  At N > 1 the global batch is batch_per_gpu * N for both arms: the CPU arm has one host, which works
    through the N per-GPU chunks one after another (its windows/s is that of one chunk; see cpu_baseline.sample)."""
    spec, res, batch, train, arp, burnin, scaling = workload(a.workload, world)
    hw = res * res
    return {"workload": a.workload, "network": spec + ".yaml", "timesteps": a.timesteps, "batch_per_gpu": batch,
            "global_batch": batch * world, "resolution": "%dx%d" % (res, res), "arp": arp, "burnin": burnin,
            "parallelism": ("dp%d (batch-sharded, NCCL allreduce of local-layer grads per timestep)" % world) if world > 1
            else "single GPU",
            "l2": "256 MiB flush buffer written between timed steps; per-step working set (state ping-pong "
                  "%.0f MB/layer) %s L2" % (2 * 2 * 4 * 32 * hw * batch / 1e6, ">" if 2 * 2 * 4 * 32 * hw * batch > 126e6 else "<")}


# --------------------------------------------------------------------------------------------------------
# CPU arm (reference arm / cpu_baseline): the reference's own classes from oracle/_ref, else the oracle port
# --------------------------------------------------------------------------------------------------------
def cpu_reference_sample(wl, T, n_fwd=1, n_train=2):
    """Times the UNMODIFIED reference (train.py:238-251 / test_radio_ml.py:140-145: iq2spiketrain -> torch.Tensor ->
    net.reset(); net.train(); net.learn(x[t], y[t]) per timestep) on a bounded sample and extrapolates linearly in T
    (BASELINE.md section 4).  Returns (windows_per_s, description, seconds, extra) or None when oracle/_ref is absent."""
    import numpy as np
    import torch
    from oracle import refshim
    if not refshim.reference_available():
        return None
    spec, res, batch, train, arp, burnin, _ = workload(wl)
    torch.set_num_threads(os.cpu_count() or 1)
    _, _, U = refshim.load_reference()
    # sample layout: 1 warm-up + n_fwd forward-only timesteps, then (training) 1 untimed first training step (builds the
    # Adam state) + n_train timed ones; the reference trains from iter >= burnin (dcll/pytorch_libdcll.py:692)
    n_s = 1 + n_fwd + ((1 + n_train) if train else 0)
    net = refshim.build_reference_net(spec, (1, res, res), batch, K_CLASSES, arp=arp, burnin=(2 + n_fwd) if train else burnin,
                                      train=train, seed=1)
    x, y = synth(batch, 1)
    spent0 = time.perf_counter()
    np.random.seed(1)
    t0 = time.perf_counter()
    with refshim.quiet():
        frames, targets = U.iq2spiketrain(x, y.numpy(), out_w=res, out_h=res, min_I=-1, max_I=1, min_Q=-1, max_Q=1,
                                          max_duration=n_s)
    inp, lab = torch.Tensor(frames), torch.Tensor(targets)                 # train.py:243-244
    enc_per_t = (time.perf_counter() - t0) / n_s
    net.reset()
    net.train() if train else net.eval()
    ts = []
    for t in range(n_s):
        t0 = time.perf_counter()
        if train:
            net.learn(x=inp[t], labels=lab[t])
        else:
            with torch.no_grad():
                net.test(x=inp[t])
        ts.append(time.perf_counter() - t0)
    t_fw = sum(ts[1:1 + n_fwd]) / n_fwd
    t_tr = sum(ts[2 + n_fwd:]) / n_train if train else 0.0
    who = "UNMODIFIED reference classes (oracle/_ref: ConvNetwork.learn/.test, data.utils.iq2spiketrain), torch %s CPU, %d threads" \
        % (torch.__version__, torch.get_num_threads())
    if train:
        window_s = enc_per_t * T + (burnin - 1) * t_fw + (T - burnin + 1) * t_tr
        desc = ("%s: %d fwd-only + %d training timesteps of %s at B=%d timed, extrapolated linearly to T=%d "
                "(%d burn-in + %d training timesteps) + encode" % (who, n_fwd, n_train, wl, batch, T, burnin - 1, T - burnin + 1))
    else:
        window_s = enc_per_t * T + T * t_fw
        desc = "%s: %d inference timesteps of %s at B=%d timed, extrapolated linearly to T=%d + encode" % (who, n_fwd, wl, batch, T)
    return batch / window_s, desc, time.perf_counter() - spent0, dict(ms_fwd_timestep=1e3 * t_fw, ms_train_timestep=1e3 * t_tr,
                                                                      ms_encode_timestep=1e3 * enc_per_t)


def cpu_port_sample(wl, T, n_fwd=1, n_train=2, reps=1):
    """Fallback when oracle/_ref is absent: the oracle port (same operator sequence: F.conv2d / autograd / torch.optim.Adam)."""
    import numpy as np
    import torch
    from oracle import dcll_oracle as O
    spec, res, batch, train, arp, burnin, _ = workload(wl)
    torch.set_num_threads(os.cpu_count() or 1)
    specs = O.make_specs(O.BUILTIN_SPECS[spec], (1, res, res), K_CLASSES, wrp=arp)
    params = O.random_params(specs, seed=1)
    net = O.OracleNet(specs, params, batch, burnin=0 if train else burnin, backend="autograd")
    x, y = synth(batch, 1)
    t_enc_n = max(8, 4 + n_fwd + n_train)
    t0 = time.perf_counter()
    cells = O.encode_cells(x.numpy(), res, res, t_start=0, max_duration=t_enc_n)
    frames = torch.from_numpy(O.cells_to_frames(cells, res, res))
    enc_per_t = (time.perf_counter() - t0) / t_enc_n
    spent0 = time.perf_counter()
    net.reset()
    with torch.no_grad():
        net.test(frames[0])                                          # untimed warm-up (allocations, oneDNN primitives)
    t_fw = t_tr = 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        with torch.no_grad():
            for i in range(n_fwd):
                net.test(frames[1 + i])
        t_fw += (time.perf_counter() - t0) / n_fwd
        if train:
            net.learn(frames[2], y)                                  # untimed: first backward builds Adam state
            t0 = time.perf_counter()
            for i in range(n_train):
                net.learn(frames[3 + i], y)
            t_tr += (time.perf_counter() - t0) / n_train
    t_fw, t_tr = t_fw / reps, t_tr / reps
    if train:
        window_s = enc_per_t * T + (burnin - 1) * t_fw + (T - burnin + 1) * t_tr
        desc = ("oracle port (F.conv2d + autograd + torch.optim.Adam, %d threads): %d fwd-only + %d training timesteps "
                "of %s at B=%d timed, extrapolated linearly to T=%d (%d burn-in + %d training timesteps) + encode"
                % (torch.get_num_threads(), n_fwd, n_train, wl, batch, T, burnin - 1, T - burnin + 1))
    else:
        window_s = enc_per_t * T + T * t_fw
        desc = ("oracle port (%d threads): %d inference timesteps of %s at B=%d timed, extrapolated linearly to T=%d + encode"
                % (torch.get_num_threads(), n_fwd, wl, batch, T))
    return batch / window_s, desc, time.perf_counter() - spent0, dict(ms_fwd_timestep=1e3 * t_fw, ms_train_timestep=1e3 * t_tr)


def cpu_sample(wl, T, n_fwd, n_train):
    """(value, description, seconds, extra, kind): the reference classes when vendored, else the port."""
    r = cpu_reference_sample(wl, T, n_fwd=n_fwd, n_train=n_train)
    if r is not None:
        return r + ("reference",)
    return cpu_port_sample(wl, T, n_fwd=n_fwd, n_train=n_train) + ("port",)


def run_reference(a):
    import torch
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    spec, res, batch, train, arp, burnin, scaling = workload(a.workload, world)
    vals = []
    big = res >= 64
    # per-GPU chunk of the workload; the single host works through the `world` chunks one after another, so its
    # windows/s is the chunk's (samples are independent; only the batch mean couples them)
    for i in range(a.warmup + a.steps):
        v, desc, _, extra, kind = cpu_sample(a.workload, a.timesteps, n_fwd=2 if big else 8, n_train=6 if big else 64)
        if i >= a.warmup:
            vals.append(v)
    v = sum(vals) / len(vals)
    unit = "windows/s"
    if world > 1:
        desc += "; N = %d: ONE host, the %d per-GPU chunks of the global batch %d are processed one after another at this rate" \
            % (world, world, batch * world)
    out = {"impl": "reference", "metric": "RadioML IQ windows/sec (DCLL %s)" % ("train" if train else "infer"),
           "value": v, "unit": unit, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": 1e3 * batch * world / v, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": config_dict(a, world),
           "cpu_baseline": {"value": v, "unit": unit, "cores": torch.get_num_threads(), "kind": kind, "sample": desc, **extra},
           "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_json(out)


# --------------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------------
def make_args(arp=0.0):
    """train.py argparse defaults (ref train.py:75-90) as the namespace ConvNetwork reads."""
    import types
    return types.SimpleNamespace(netscale=1.0, alpha=0.92, alphas=0.85, alpharp=0.65, arp=arp, lc_ampl=0.5, random_tau=True)


def build_net(wl, world=1):
    import numpy as np
    import torch
    from snn_modulation_classification_b200 import networks as N
    spec, res, batch, train, arp, burnin, _ = workload(wl, world)
    torch.manual_seed(1)
    np.random.seed(1)
    kw = dict(loss=torch.nn.SmoothL1Loss, opt=torch.optim.Adam, opt_param={"betas": [0.0, 0.95], "weight_decay": 10.0},
              learning_rates=[1e-6]) if train else dict(loss=None, opt=None, opt_param={}, learning_rates=None)
    net = N.ConvNetwork(make_args(arp), (1, res, res), batch, N.load_network_spec(spec), K_CLASSES,
                        act=torch.nn.Sigmoid(), burnin=burnin, **kw)
    net.reset(True)
    return net


def sample_index(n):
    """DUMP_SAMPLE sorted distinct indices into n > DUMP_SAMPLE elements, the same for every run: one index drawn from a
    fixed seed inside each of DUMP_SAMPLE equal strata at the head of the flat array (its last n % DUMP_SAMPLE elements are
    not sampled)."""
    import numpy as np
    stride = n // DUMP_SAMPLE
    return np.arange(DUMP_SAMPLE) * stride + np.random.default_rng(0).integers(0, stride, DUMP_SAMPLE)


def step_outputs(net, clout, train):
    """{name: float32 array} of what a window hands back to its caller: the class votes clout [T, layers, B], and per layer
    the parameters and, after a training window, the neuron state.  (Inference windows leave no state to compare: the
    16x16 multi-timestep kernel keeps it on chip and returns only the votes.)  Arrays above DUMP_SAMPLE elements become
    the sample at sample_index."""
    import torch
    arrays = {"clout": clout}
    for i, sl in enumerate(net.dcll_slices):
        lay = sl.dclllayer
        arrays["l%d_weight" % i], arrays["l%d_bias" % i] = lay.i2h.weight, lay.i2h.bias
        if lay.output_layer:
            arrays["l%d_output_weight" % i], arrays["l%d_output_bias" % i] = lay.output_.weight, lay.output_.bias
        if train:
            for field, t in zip(lay.i2h.state._fields, lay.i2h.state):
                arrays["l%d_%s" % (i, field)] = t
    out, index = {}, {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            if t.numel() not in index:
                index[t.numel()] = torch.from_numpy(sample_index(t.numel())).to(t.device)
            t, name = t.reshape(-1)[index[t.numel()]], name + "_sample"
        out[name] = t.float().cpu().numpy()
    return out


def _event_timed(fn, steps, flush=None):
    import torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps


def other_workloads(flush):
    """Short runs of the other BASELINE.json configs through the same public API (driver-visible; each entry names its
    configuration).  1 warm-up + 2 timed windows each, CUDA events, L2 flushed between windows."""
    import numpy as np
    import torch
    from snn_modulation_classification_b200 import networks as N
    from snn_modulation_classification_b200.data.utils import iq2spiketrain
    from snn_modulation_classification_b200.quant import enable_quantized_weights
    res_out = []

    def train_net(spec, im, batch, K, burnin, arp=0.0):
        torch.manual_seed(1)
        np.random.seed(1)
        net = N.ConvNetwork(make_args(arp), im, batch, N.load_network_spec(spec), K, act=torch.nn.Sigmoid(),
                            loss=torch.nn.SmoothL1Loss, opt=torch.optim.Adam,
                            opt_param={"betas": [0.0, 0.95], "weight_decay": 10.0}, learning_rates=[1e-6], burnin=burnin)
        net.reset(True)
        return net.set_precision("bf16x3")

    def record(name, cfg, B, T, ms, **extra):
        res_out.append(dict(name=name, config=cfg, windows_per_s=B / (ms / 1e3), ms_per_window_batch=ms,
                            sample_timesteps_per_s=B * T / (ms / 1e3), **extra))

    # configs[1]: mnist_conv.yaml on synthetic 28x28 Bernoulli spike trains (data/utils.py:23-31: rate = gain*pixel/1000)
    B, T = 128, 500
    net = train_net("mnist_conv", (1, 28, 28), B, 10, 50)
    g = torch.Generator().manual_seed(1)
    img = torch.rand(B, 1, 28, 28, generator=g)
    frames = (torch.rand(T, B, 1, 28, 28, generator=g) < img * (100.0 / 1000.0)).float().cuda()
    y10 = torch.zeros(B, 10).scatter_(1, torch.randint(0, 10, (B,), generator=g).unsqueeze(-1), 1).cuda()

    def step_mnist():
        net.reset()
        net.learn_window(frames, y10)
    step_mnist()
    record("mnist_conv_train_28x28_B128", "BASELINE configs[1]: mnist_conv.yaml train, B=128, T=500, dense Bernoulli frames, K=10",
           B, T, _event_timed(step_mnist, 2, flush), tensor_core_layers=[bool(s.dclllayer.i2h.tensor_core_ok()) for s in net.dcll_slices])
    del net, frames

    # configs[2]: radio_ml_conv_ref.yaml as a 7-layer DCLL spec with int8-quantised weights
    B, T = 32, 64
    net = train_net("radio_ml_conv_ref", (1, 128, 128), B, K_CLASSES, 16)
    enable_quantized_weights(net)
    x, y = synth(B, 1)
    x, y = x.cuda(), y.cuda()
    enc = dict(out_w=128, out_h=128, min_I=-1, max_I=1, min_Q=-1, max_Q=1, max_duration=T, as_cells=True)

    def step_q():
        cells, _ = iq2spiketrain(x, y, **enc)
        net.reset()
        net.learn_window(cells, y)
    step_q()
    record("radio_ml_conv_ref_quant_train_128x128_B32", "BASELINE configs[2]: radio_ml_conv_ref.yaml (7 layers, 1x3 kernels, 64 ch), "
           "int8-quantised weights, train, B=32, T=64, 128x128", B, T, _event_timed(step_q, 2, flush),
           tensor_core_layers=[bool(s.dclllayer.i2h.tensor_core_ok()) for s in net.dcll_slices])
    del net

    # script geometry (scripts/train_radio_ml.sh): 16x16, B=512, arp=1, burnin=20
    for name, B, T, train, arp, burnin in (("radio_ml_conv_train_16x16_B512_arp", 512, 256, True, 1.0, 20),
                                           ("radio_ml_conv_infer_16x16_B4096", 4096, 256, False, 1.0, 20),
                                           ("radio_ml_conv_infer_16x16_B65536", 65536, 64, False, 1.0, 20),
                                           ("radio_ml_conv_infer_16x16_B256", 256, 512, False, 1.0, 20)):
        WORKLOADS["_tmp"] = ("radio_ml_conv", 16, B, train, arp, burnin)
        net = build_net("_tmp").set_precision("bf16x3")
        x, y = synth(B, 1)
        x, y = x.cuda(), y.cuda()
        enc = dict(out_w=16, out_h=16, min_I=-1, max_I=1, min_Q=-1, max_Q=1, max_duration=T, as_cells=True)

        def step_s():
            cells, _ = iq2spiketrain(x, y, **enc)
            net.reset()
            if train:
                net.learn_window(cells, y)
            else:
                net.test_window(cells)
                net.dcll_slices[-1].clout.vote_device(K_CLASSES)
        step_s()
        what = "train (scripts/train_radio_ml.sh geometry)" if train else "BASELINE configs[3] inference sweep point (multi-timestep kernel + device vote)"
        record(name, "radio_ml_conv.yaml %s, 16x16, B=%d, T=%d, arp=%g" % (what, B, T, arp), B, T, _event_timed(step_s, 2, flush))
        del net
    WORKLOADS.pop("_tmp", None)
    torch.cuda.empty_cache()
    return res_out


def config5_line(world, rank, flush, T=128):
    """radio_ml_conv data-parallel training at global batch 8192 (BASELINE.json configs[4]), 16x16, T timesteps, bf16x3:
    1 warm-up + 2 timed windows, barrier + device events, max over ranks.  Collective on every rank."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from snn_modulation_classification_b200.data.utils import iq2spiketrain
    name = "radio_ml_conv_train_dp_global8192_16x16"
    spec, res, batch, train, arp, burnin, scaling = workload(name, world)
    net = build_net(name, world).set_precision("bf16x3")
    if world > 1:
        for p in net.state_dict().values():
            dist.broadcast(p, 0)
    x, y = synth(batch, 100 + rank)
    x, y = x.cuda(), y.cuda()
    enc = dict(out_w=res, out_h=res, min_I=-1, max_I=1, min_Q=-1, max_Q=1, max_duration=T, as_cells=True)

    def step():
        cells, _ = iq2spiketrain(x, y, **enc)
        net.reset()
        if world > 1:
            net.learn_window_dp(cells, y)
        else:
            net.learn_window(cells, y)
    np.random.seed(1)
    step()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([_event_timed(step, 2, flush)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    del net
    torch.cuda.empty_cache()
    return {"workload": name, "global_batch": batch * world, "batch_per_gpu": batch, "n_gpus": world, "timesteps": T,
            "resolution": "16x16", "scaling": scaling, "windows_per_s": batch * world / (ms / 1e3), "ms_per_window_batch": ms,
            "sample_timesteps_per_s": batch * world * T / (ms / 1e3),
            "note": "whole-job windows/s at T=%d (not extrapolated to 1024); %s" % (
                T, "NCCL all-reduce of the local-layer gradient buckets per timestep inside dcll_net_window_dp" if world > 1
                else "single GPU: no collective")}


def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.data.utils import iq2spiketrain

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    spec, res, batch, train, arp, burnin, scaling = workload(a.workload, world)
    T = a.timesteps
    net = build_net(a.workload, world)
    net.set_precision(a.precision)
    tc = any(sl.dclllayer.i2h.tensor_core_ok() for sl in net.dcll_slices)
    # layers whose trace operand is one fp16 value (2 products per MAC, 2-byte operand image) in f16x2 mode
    f16_layers = [a.precision == "f16x2" and sl.dclllayer.i2h.f16_ok(*[int(v) for v in sl.dclllayer.im_dims])
                  for sl in net.dcll_slices]
    if world > 1:                                   # identical replicas: broadcast rank 0's parameters
        for p in net.state_dict().values():
            dist.broadcast(p, 0)
    x, y = synth(batch, 1 + rank)
    x_pin, y_pin = x.pin_memory(), y.pin_memory()
    x_dev, y_dev = x.cuda(), y.cuda()
    pred_pin = torch.empty(batch, dtype=torch.int32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    enc = dict(out_w=res, out_h=res, min_I=-1, max_I=1, min_Q=-1, max_Q=1, max_duration=T, as_cells=True)

    def run_window(cells, labels):
        net.reset()
        if not train:
            return net.test_window(cells)
        if world > 1:
            return net.learn_window_dp(cells, labels)
        return net.learn_window(cells, labels)

    last = {}

    def step_device():
        cells, _ = iq2spiketrain(x_dev, y_dev, **enc)
        last["clout"] = run_window(cells, y_dev)

    def step_e2e():
        xd = x_pin.to("cuda", non_blocking=True)
        yd = y_pin.to("cuda", non_blocking=True)
        cells, _ = iq2spiketrain(xd, yd, **enc)
        run_window(cells, yd)
        pred = net.dcll_slices[-1].clout.vote_device(K_CLASSES)
        pred_pin.copy_(pred, non_blocking=True)

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(steps):
            flush.zero_()                          # L2 flush between timed iterations (256 MiB > 126 MB L2)
            fn()
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    np.random.seed(1)
    for _ in range(a.warmup):
        step_device()
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    _lib.lib.dcll_launch_count(1)
    _lib.check(_lib.lib.dcll_profile_enable(a.profile_every))
    ms = timed(step_device, a.steps)
    launches = int(_lib.lib.dcll_launch_count(0))
    prof = _lib.profile_read()
    _lib.check(_lib.lib.dcll_profile_enable(0))
    dumped = step_outputs(net, last["clout"], train) if a.dump_outputs and rank == 0 else None
    ms_e2e = timed(step_e2e, a.steps)
    clocks = sampler.stop() if sampler else None
    # BASELINE.json configs[4]: data-parallel training at GLOBAL batch 8192 (8192 / N windows per GPU; 16x16 script geometry, which
    # fits any N), a short window on every rank so that the line is driver-visible at each N of the scaling run
    cfg5 = None
    n_layers = len(net.dcll_slices)
    if not a.no_extras and a.workload == DEFAULT and 8192 % world == 0:
        net = None
        torch.cuda.empty_cache()
        cfg5 = config5_line(world, rank, flush)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * batch * a.steps / (ms / 1e3)
    e2e = world * batch * a.steps / (ms_e2e / 1e3)
    pk = peaks()
    hw = res * res
    per_class = {}
    for (name, layer), (tms, n) in sorted(prof.items()):
        per_class["%s[l%d]" % (name, layer)] = {"avg_ms": tms / n, "samples": n}

    def avg(name, layer):
        tms, n = prof.get((name, layer), (0.0, 0))
        return (tms / n if n else None), n

    # ---- roofline.  Kernel classes and their algorithmic work per launch (DESIGN.md section 4):
    #   wgrad[l]       wgrad_tc_kernel (bracket minus the reduce_adam launch inside it)   2*Cin*49*Cout*H'W'*B FLOP   tensor
    #   conv_fwd[l]    conv_mma(2)_kernel (bracket minus the trace pass inside it)        the same FLOP              tensor
    #   trace[l]       trace_image_kernel                                                  24 B per state element     hbm
    #   readout_fwd[l] readout_tc + finish    pv (4 B/elem) + Wo (4*Ktot*F)               hbm
    #   readout_bwd[l] g_u sweep (+ output_ gradient/Adam on the last layer)              hbm
    # `roofline` is quoted on the class with the LARGEST share of the sampled step; the others follow in roofline.kernels.
    adam_ms, _ = avg("adam", 0)
    kernels = []
    conv_flops = lambda cin: 2.0 * cin * 49 * 32 * hw * batch
    for l in range(n_layers):
        cin = 1 if l == 0 else 32
        elems_in, elems_out = cin * hw * batch, 32 * hw * batch
        ktot = K_CLASSES * (2 if l == n_layers - 1 else 1)
        c_ms, c_n = avg("conv_fwd", l)
        t_ms, _ = avg("trace", l)
        if c_ms:
            k_ms = c_ms - (t_ms or 0.0)
            kernels.append(dict(kernel="conv_fwd[l%d] (%s)" % (l, "tcgen05 conv_mma/conv_mma2" if tc else "FP32 FMA conv_fwd_kernel"),
                                bound="tensor", ms=k_ms, samples=c_n, work=conv_flops(cin), unit="TFLOP/s", products=2 if f16_layers[l] else 3,
                                achieved=conv_flops(cin) / (k_ms * 1e-3) / 1e12, peak=pk["tensor"]))
        if t_ms:
            # bytes: x in (4 B dense; one cell per sample when fed cells), eps0/eps1 read + written, operand image written
            img = (2 if f16_layers[l] else 4) * (8 if cin == 1 else cin) / cin   # single channel: 8 column shifts per position; hi + lo, or one fp16
            byt = elems_in * ((0 if l == 0 else 4) + 16 + img)
            kernels.append(dict(kernel="trace[l%d] (trace_image_kernel)" % l, bound="hbm", ms=t_ms, samples=c_n, work=byt,
                                unit="GB/s", achieved=byt / (t_ms * 1e-3) / 1e9, peak=pk["hbm"]))
        w_ms, w_n = avg("wgrad", l)
        if w_ms:
            k_ms = w_ms - (adam_ms or 0.0)
            kernels.append(dict(kernel="wgrad[l%d] (%s)" % (l, "tcgen05 wgrad_tc2p/wgrad_tc" if tc else "FP32 FMA wgrad_kernel"), bound="tensor",
                                ms=k_ms, samples=w_n, work=conv_flops(cin), unit="TFLOP/s", products=2 if f16_layers[l] else 3,
                                achieved=conv_flops(cin) / (k_ms * 1e-3) / 1e12, peak=pk["tensor"]))
        r_ms, r_n = avg("readout_fwd", l)
        if r_ms:
            byt = 4.0 * elems_out + 4.0 * ktot * 32 * hw
            kernels.append(dict(kernel="readout_fwd[l%d] (readout_tc + finish)" % l, bound="hbm", ms=r_ms, samples=r_n, work=byt,
                                unit="GB/s", achieved=byt / (r_ms * 1e-3) / 1e9, peak=pk["hbm"]))
        b_ms, b_n = avg("readout_bwd", l)
        if b_ms:
            byt = 8.0 * elems_out + 4.0 * K_CLASSES * 32 * hw            # pv in, g_u out, Wo once
            if l == n_layers - 1:
                byt += 4.0 * elems_out + 6 * 4.0 * K_CLASSES * 32 * hw   # pv again, Wout/m/v read + written
            kernels.append(dict(kernel="readout_bwd[l%d]" % l, bound="hbm", ms=b_ms, samples=b_n, work=byt, unit="GB/s",
                                achieved=byt / (b_ms * 1e-3) / 1e9, peak=pk["hbm"]))
    for k in kernels:
        k["frac"] = k["achieved"] / k["peak"]
        if k["bound"] == "tensor" and tc:
            k["frac_executed"] = k["products"] * k["frac"]   # split operands: 3 (bf16x3) or 2 (f16x2) products per algorithmic MAC
    # share per kernel CLASS (layers of the same shape summed): the dominant class is the one the step spends most time in
    cls = {}
    for k in kernels:
        name = k["kernel"].split("[")[0]
        cls.setdefault(name, []).append(k)
    step_ms = sum(k["ms"] for k in kernels) or 1.0
    dom_name = max(cls, key=lambda n_: sum(k["ms"] for k in cls[n_])) if cls else None
    roofline = None
    if dom_name:
        grp = [k for k in cls[dom_name]]
        big = max(grp, key=lambda k: k["ms"])           # quoted on the largest launch of the class (a 32->32 layer)
        roofline = {"kernel": big["kernel"], "bound": big["bound"], "achieved": big["achieved"], "peak": big["peak"],
                    "unit": big["unit"], "frac": big["frac"],
                    # dram bytes per launch are an ncu quantity; they are not measured inside this run (profiles/*ncu*.txt
                    # of the round hold the `ncu --set full` capture of this kernel)
                    "traffic": None,
                    "peak_source": "%s %s (MEASURED_PEAKS.json)" % (pk["src"], "bf16 dense sustained" if big["bound"] == "tensor" else "HBM copy bandwidth"),
                    "avg_launch_ms": big["ms"], "launches_sampled": big["samples"],
                    "algorithmic_work_per_launch": big["work"],
                    "class_share_of_step": sum(k["ms"] for k in grp) / step_ms,
                    "frac_executed": big.get("frac_executed"),
                    "note": ("achieved counts ALGORITHMIC conv FLOPs (one product per MAC); the split-operand modes execute `products` "
                             "16-bit products per MAC (3 in bf16x3, 2 in f16x2; frac_executed = share of the tensor peak actually issued)"
                             if tc and big["bound"] == "tensor" else None),
                    "kernels": [{kk: (round(v, 6) if isinstance(v, float) else v) for kk, v in k.items()} for k in
                                sorted(kernels, key=lambda k: -k["ms"])]}

    out = {"metric": "RadioML IQ windows/sec (DCLL %s)" % ("train" if train else "infer"), "value": value,
           "unit": "windows/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
           "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
           "dtype": ({"bf16x3": "bf16x3 (split-bf16 operands on tcgen05, 3 products per MAC, fp32 accumulate; traces/neuron/update fp32)",
                      "f16x2": "f16x2 (fp16 traces x split-fp16 weights / local gradients on tcgen05, 2 products per MAC, fp32 accumulate; "
                               "layer 0 split-bf16 x3; traces/neuron/update fp32)"}[a.precision] if tc else "f32"),
           "precision": a.precision, "data": "synthetic", "config": config_dict(a, world),
           "sample_timesteps_per_s": value * T,
           "model_tflops": value * T * flops_per_sample_timestep(res, train) / 1e12,
           "e2e": {"value": e2e, "unit": "windows/s", "ms_per_step": ms_e2e / a.steps,
                   "h2d_bytes_per_step": int(x_pin.numel() * 4 + y_pin.numel() * 4),
                   "d2h_bytes_per_step": int(pred_pin.numel() * 4)},
           "gpu_launches": launches, "roofline": roofline, "kernel_ms": per_class, "clocks": clocks}
    if cfg5 is not None:
        out["dp_global_batch_8192"] = cfg5
    if world == 1 and a.precision != "fp32" and not a.no_extras:
        net = build_net(a.workload, world)
        net.set_precision(a.precision)
        # BASELINE.json configs[0] says FP32: the same workload in the FP32-exact parity mode (CUDA-core FMA kernels), whole
        # windows at the full T, 1 warm-up + 2 timed
        net.set_precision("fp32")
        step_device()
        ms32 = _event_timed(step_device, 2, flush)
        out["fp32_mode"] = {"value": batch / (ms32 / 1e3), "unit": "windows/s", "ms_per_step": ms32, "steps": 2, "timesteps": T,
                            "note": "FP32-exact parity mode (every tolerance of DESIGN.md section 2 holds), same workload"}
        if a.precision == "f16x2":
            # the three-product split-bf16 mode (membrane within ~1e-5 of its scale instead of ~2e-4), same workload, 1 + 2 windows
            net.set_precision("bf16x3")
            step_device()
            msb = _event_timed(step_device, 2, flush)
            out["bf16x3_mode"] = {"value": batch / (msb / 1e3), "unit": "windows/s", "ms_per_step": msb, "steps": 2, "timesteps": T,
                                  "note": "split-bf16 x3 tensor-core mode, same workload"}
        net = None                                   # free the 128x128 state before the other workloads allocate theirs
        torch.cuda.empty_cache()
        out["other_workloads"] = other_workloads(flush)
    if world == 1 and not a.no_cpu:
        big = res >= 64
        # ~10-25 s of CPU work on the bounded sample (16 host cores: ~0.5 s / 0.7 s per 128x128 timestep)
        v, desc, spent, extra, kind = cpu_sample(a.workload, T, n_fwd=4 if big else 16, n_train=12 if big else 256)
        out["cpu_baseline"] = {"value": v, "unit": "windows/s", "cores": torch.get_num_threads(), "kind": kind,
                               "sample": desc, "seconds": spent, **extra}
    if dumped is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    emit_json(out)
    if world > 1:
        dist.destroy_process_group()


class _StdoutGuard:
    """Everything libraries print to fd 1 while the benchmark runs (e.g. NCCL's version banner) goes to stderr;
    only the final JSON line reaches the real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.saved, (line + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


_GUARD = None


def emit_json(obj):
    line = json.dumps(obj)
    if _GUARD is not None:
        _GUARD.emit(line)
    else:
        print(line, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT, choices=sorted(WORKLOADS))
    ap.add_argument("--timesteps", type=int, default=1024)
    ap.add_argument("--profile-every", type=int, default=31, dest="profile_every")
    ap.add_argument("--no-cpu", action="store_true", dest="no_cpu")
    ap.add_argument("--no-extras", action="store_true", dest="no_extras",
                    help="skip the fp32_mode and other_workloads legs (quick profiling runs)")
    ap.add_argument("--precision", default="f16x2", choices=["fp32", "bf16x3", "f16x2"],
                    help="fp32: FP32-exact parity mode on the FMA pipe; bf16x3: tcgen05, split-bf16 operands, 3 products per MAC; "
                         "f16x2 (headline mode): tcgen05, fp16 traces against split-fp16 weights / gradients, 2 products per MAC")
    ap.add_argument("--burnin", type=int, default=None, help="override the workload's burn-in (profiling runs)")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (float32; large arrays as a seeded sample)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to the B200 arm")
    if a.burnin is not None:
        w = list(WORKLOADS[a.workload])
        w[5] = a.burnin
        WORKLOADS[a.workload] = tuple(w)
    global _GUARD
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    with _StdoutGuard() as g:
        _GUARD = g
        if a.impl == "reference":
            run_reference(a)
        else:
            run_b200(a)
    _GUARD = None


if __name__ == "__main__":
    main()
