#!/usr/bin/env python
"""Inference sweep at 16x16 (SURVEY 8(d) config 4): windows/s of ConvNetwork.test_window over B x T.

    python tools/infer_sweep.py > profiles/r01_infer_sweep_16x16.jsonl
    python tools/infer_sweep.py --precision f16x2 --B 256 4096 65536 --T 256
    python tools/infer_sweep.py --precision f16x2 --path per_timestep --B 4096 --T 256

One JSON line per (B, T): device-resident IQ records -> iq2spiketrain (cells) -> test_window (dcll_infer_stack16 +
dcll_conv_readout_rows in bf16x3 mode, or the mode of --precision) -> device vote.  CUDA events, 1 warm-up + 3 timed
windows, L2 flushed between.  --path per_timestep times the per-timestep kernels (dcll_net_window) on the same input
instead, --path stack the multi-timestep kernel whether or not test_window would choose it.
--check_votes: where the multi-timestep kernel runs, one more window of each path on the timed input reports the share of
equal votes.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
from snn_modulation_classification_b200.data.utils import iq2spiketrain


def run(B, T, precision="bf16x3", path="auto", check_votes=False):
    bench.WORKLOADS["sweep"] = ("radio_ml_conv", 16, B, False, 1.0, 20)
    net = bench.build_net("sweep")
    net.set_precision(precision)
    x, y = bench.synth(B, 1)
    x, y = x.cuda(), y.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    enc = dict(out_w=16, out_h=16, min_I=-1, max_I=1, min_Q=-1, max_Q=1, max_duration=T, as_cells=True)

    def step(how=path):
        cells, _ = iq2spiketrain(x, y, **enc)
        net.reset()
        if how == "auto":
            net.test_window(cells)
        elif how == "stack":
            net._run_stack16(cells)
        else:
            net._run_window(cells, None, False)
        return net.dcll_slices[-1].clout.vote_device(bench.K_CLASSES)

    np.random.seed(1)
    step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 3
    e0.record()
    for _ in range(steps):
        flush.zero_()
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    stack = path == "stack" or (path == "auto" and bool(net._stack16_ok(iq2spiketrain(x, y, **enc)[0])))
    r = {"B": B, "T": T, "precision": precision, "ms_per_window_batch": ms, "windows_per_s": B / (ms / 1e3),
         "sample_timesteps_per_s": B * T / (ms / 1e3), "multi_timestep_kernel": stack}
    if stack and check_votes:
        np.random.seed(1)           # the spike encoding draws from numpy: the same cells for both paths
        va = step("stack")
        np.random.seed(1)
        vb = step("per_timestep")
        r["votes_equal_to_per_timestep"] = float((va == vb).float().mean())
    return r


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16x3", "f16x2"])
    ap.add_argument("--path", default="auto", choices=["auto", "stack", "per_timestep"],
                    help="auto: test_window's choice; stack / per_timestep: that path")
    ap.add_argument("--check_votes", action="store_true", help="compare the votes of both paths on the timed input")
    ap.add_argument("--B", type=int, nargs="+", help="batch sizes (default: the full sweep)")
    ap.add_argument("--T", type=int, nargs="+", help="window lengths (default: the full sweep)")
    args = ap.parse_args()
    for B in args.B or (256, 1024, 4096, 16384, 65536):
        for T in args.T or (64, 256, 512):
            if args.B is None and args.T is None and B * T > 65536 * 256:      # keep the sweep within a few GPU-minutes
                continue
            print(json.dumps(run(B, T, args.precision, args.path, args.check_votes)), flush=True)
    if args.B is None and args.T is None:
        print(json.dumps(run(4096, 256, "fp32")), flush=True)   # per-timestep FP32 path for comparison
