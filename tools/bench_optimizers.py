#!/usr/bin/env python
"""learn_window throughput per optimizer: the radio_ml_conv stack at 128x128, B = 64, T = 128, f16x2, trained with
torch.optim.Adam and with each optimizer the device applies besides it (AdamW, Adamax, NAdam, RAdam), all built as train.py
builds them (betas (0, 0.95), weight_decay 10; optimizer2 with lr 1e-4).  One JSON line per optimizer: the median of three
timed windows (CUDA events, after one warm-up window), with the card's name and power limit.

    python tools/bench_optimizers.py [--windows 3] [--T 128]

The update kernels move the same bytes for every rule (two float32 state tensors per parameter), so each rule is expected to
land within a few percent of Adam.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
from snn_modulation_classification_b200 import networks as N
from snn_modulation_classification_b200.data.utils import iq2spiketrain


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, limit = (v.strip() for v in out[0].split(","))
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(), None


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--T", type=int, default=128)
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--res", type=int, default=128)
    a = ap.parse_args(argv)
    name, limit = card()
    x, y = bench.synth(a.B, seed=1)
    np.random.seed(1)
    cells, _ = iq2spiketrain(x, y, out_w=a.res, out_h=a.res, max_duration=a.T, as_cells=True)
    y = y.cuda()
    for optim_type in ("Adam", "AdamW", "Adamax", "NAdam", "RAdam"):
        torch.manual_seed(1)
        np.random.seed(1)
        net = N.ConvNetwork(bench.make_args(0.0), (1, a.res, a.res), a.B, N.load_network_spec("radio_ml_conv"), bench.K_CLASSES,
                            act=torch.nn.Sigmoid(), loss=torch.nn.SmoothL1Loss, opt=getattr(torch.optim, optim_type),
                            opt_param={"betas": [0.0, 0.95], "weight_decay": 10.0}, learning_rates=[1e-6], burnin=50)
        net.reset(True)
        net.set_precision("f16x2")
        net.learn_window(cells, y)                                       # warm-up
        ms = []
        for _ in range(a.windows):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            net.learn_window(cells, y)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        w = net.dcll_slices[-1].dclllayer.i2h.weight
        print(json.dumps({"optim": optim_type, "res": a.res, "B": a.B, "T": a.T, "precision": "f16x2",
                          "window_ms_median": float(np.median(ms)), "window_ms": ms,
                          "windows_per_s": 1000.0 / float(np.median(ms)), "finite": bool(torch.isfinite(w).all()),
                          "gpu": name, "power_limit": limit}), flush=True)
        del net
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
