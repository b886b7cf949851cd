"""The 16x16 multi-timestep inference kernel (dcll_infer_stack16) in 'f16x2' and with quantised weights, and the
--precision option of the CLIs.

In 'f16x2' the kernel's 32 -> 32 layers take the operand form of the per-timestep f16x2 forward (one fp16 trace plane
scaled by 2^a_exp, fp16 {hi,lo} weight image scaled by 2^w_exp); with quantised weights it reads the images the weight
sync left in place.  Each mode is held to the bounds the bf16x3 stack kernel meets against its per-timestep path
(test_gpu_tensorcore.py), and 'f16x2' additionally to the free-running bounds of test_gpu_f16x2.py against the FP32 oracle.
The CLI parsing tests run without a GPU; everything else needs a B200 (pytest -m gpu).
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import dcll_oracle as O
from util_build import build_pair

FLIP_TOL = 1e-3        # stated flip-rate bound of the headline mode (test_gpu_f16x2.py)
B, K, T, W = 12, 24, 37, 16
STACK = {"f16x2": "infer_stack16_kernel<true>", "bf16x3": "infer_stack16_kernel<false>"}


def _cells(Bn=B, Tn=T, Wn=W, seed=9):
    from snn_modulation_classification_b200.data.utils import iq2spiketrain
    g = torch.Generator().manual_seed(seed)
    xs = (torch.randn(Bn, 2, 1, 1024, generator=g) * 0.4).float()
    y = O.to_one_hot(torch.randint(0, K, (Bn,), generator=g), K)
    np.random.seed(1)
    return iq2spiketrain(xs, y, out_w=Wn, out_h=Wn, max_duration=Tn, as_cells=True)


def _net(mode, arp=0.0, quantized=False, **kw):
    from snn_modulation_classification_b200 import quant
    net, onet = build_pair("radio_ml_conv", (1, W, W), B, K, arp=arp, **kw)
    net.set_precision(mode)
    if quantized:
        quant.enable_quantized_weights(net)
    return net, onet


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key.replace(" ", "") for e in prof.key_averages()}


def _assert_stack_matches_per_step(a, b, tgt, arp):
    """a ran the stack kernel, b the per-timestep kernels of the same mode on the same cells (bounds of
    test_gpu_tensorcore.py::test_multi_timestep_stack_kernel_matches_per_step_path)."""
    for i, (sa, sb) in enumerate(zip(a.dcll_slices, b.dcll_slices)):
        ea, eb = sa.dclllayer.i2h.state, sb.dclllayer.i2h.state
        assert float((ea.eps1 != eb.eps1).float().mean()) <= 1e-3, i
        if arp > 0:
            assert float((ea.arp - eb.arp).abs().gt(1e-5).float().mean()) <= 1e-3, i
        ca, cb = np.array(sa.clout), np.array(sb.clout)
        assert ca.shape == cb.shape == (T, B)
        assert (ca == cb).mean() >= 0.995, (i, (ca == cb).mean())
        assert sa.iter == sb.iter == T
    assert torch.equal(a.dcll_slices[0].dclllayer.i2h.state.eps1, b.dcll_slices[0].dclllayer.i2h.state.eps1)
    assert a.accuracy(tgt) == b.accuracy(tgt)


def _stack16_expected(net, x):
    """Restatement of the conditions under which test_window takes dcll_infer_stack16."""
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import SpikeCells
    if not isinstance(x, SpikeCells) or len(net.dcll_slices) != 3:
        return False
    modes = []
    for i, s in enumerate(net.dcll_slices):
        lay, c = s.dclllayer, s.dclllayer.i2h
        ok = (tuple(int(v) for v in lay.im_dims) == (16, 16) and c.kernel_size == (7, 7) and c.padding == (3, 3)
              and tuple(lay.pooling) == (1, 1) and c.out_channels == 32 and c.in_channels == (1 if i == 0 else 32)
              and c.precision in ("bf16x3", "f16x2") and c.state.eps0.shape[0] == x.cells.shape[1])
        if not ok:
            return False
        modes.append(c.precision)
    return modes[1] == modes[2] and (modes[1] != "f16x2" or x.cells.shape[1] <= 4096)


# ------------------------------------------------------------------------------------------------------------------------
# 1 + 2: stack kernel against the per-timestep path of the same network (f16x2, quantised bf16x3 / f16x2)
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("arp", [0.0, 1.0])
def test_f16x2_stack_kernel_matches_per_step_path_and_oracle(arp):
    cells, tgt = _cells()
    a, onet = _net("f16x2", arp, train=False)
    b, _ = _net("f16x2", arp, train=False)
    for n in (a, b, onet):
        n.reset()
    assert a._stack16_ok(cells)
    a._run_stack16(cells, chunk=5)                    # 8 launches incl. a ragged last chunk
    b._run_window(cells, None, False)
    _assert_stack_matches_per_step(a, b, tgt, arp)
    # free-running against the FP32 oracle: one launch over the window keeps pv of every timestep (spike <=> pv > 1/2)
    frames = cells.dense().cpu()
    c, _ = _net("f16x2", arp, train=False)
    c.reset()
    c._run_stack16(cells, chunk=T)
    pv = [p.view(T, B, 32, W, W).cpu() for p in c._s16["pv"]]
    flips = np.zeros(2)
    for t in range(T):
        onet.test(frames[t])
        for i in range(2):
            flips[i] += float(((pv[i][t] > 0.5).float() != onet.last[i].spikes).float().mean())
    assert (flips / T).max() <= FLIP_TOL, flips / T
    # votes: the bound of test_gpu_f16x2.py where the per-timestep f16x2 path meets it, else that path's own agreement
    # (with arp = 1 it measured 0.977 on this input) less the 0.005 the two paths may differ by
    for i, (sc, sb) in enumerate(zip(c.dcll_slices, b.dcll_slices)):
        ref = np.array(onet.clout[i])
        agree, agree_b = (np.array(sc.clout) == ref).mean(), (np.array(sb.clout) == ref).mean()
        assert agree >= min(0.98, agree_b - 0.005), (i, agree, agree_b)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["bf16x3", "f16x2"])
def test_quantized_stack_kernel_matches_per_step_path(mode):
    cells, tgt = _cells()
    a, _ = _net(mode, 1.0, quantized=True, train=False)
    b, _ = _net(mode, 1.0, quantized=True, train=False)
    a.reset()
    b.reset()
    assert a._stack16_ok(cells)
    names = _kernel_names(lambda: a._run_stack16(cells, chunk=5))
    assert any(STACK[mode] in k for k in names), sorted(names)
    b._run_window(cells, None, False)
    _assert_stack_matches_per_step(a, b, tgt, 1.0)


# ------------------------------------------------------------------------------------------------------------------------
# 3: which networks take the kernel, and which instantiation runs
# ------------------------------------------------------------------------------------------------------------------------
def _pooled_spec():
    from snn_modulation_classification_b200 import networks as N
    spec = [dict(out_channels=32, kernel_size=7, padding=3, pooling=1) for _ in range(2)] + \
           [dict(out_channels=32, kernel_size=7, padding=3, pooling=2)]
    O.BUILTIN_SPECS["stack16_pooled"] = spec
    N.BUILTIN_SPECS["stack16_pooled"] = spec


def _per_element_tau(net):
    with torch.no_grad():
        net.dcll_slices[1].dclllayer.i2h.alpha[0, 0, 0] += 1e-3


def _mixed(net):
    net.dcll_slices[2].dclllayer.i2h.precision = "bf16x3"
    net.dcll_slices[2].dclllayer.i2h._wt_key = None


CASES = {   # name: (mode, quantized, image width, spec, edit, dense input, kernel expected[, batch])
    "f16x2": ("f16x2", False, 16, "radio_ml_conv", None, False, "f16x2"),
    "bf16x3": ("bf16x3", False, 16, "radio_ml_conv", None, False, "bf16x3"),
    "f16x2_quantized": ("f16x2", True, 16, "radio_ml_conv", None, False, "f16x2"),
    "bf16x3_quantized": ("bf16x3", True, 16, "radio_ml_conv", None, False, "bf16x3"),
    "fp32": ("fp32", False, 16, "radio_ml_conv", None, False, None),
    "f16x2_8x8": ("f16x2", False, 8, "radio_ml_conv", None, False, None),
    "f16x2_pooled": ("f16x2", False, 16, "stack16_pooled", None, False, None),
    "f16x2_per_element_tau": ("f16x2", False, 16, "radio_ml_conv", _per_element_tau, False, None),
    "f16x2_dense_input": ("f16x2", False, 16, "radio_ml_conv", None, True, None),
    "mixed_hidden_forms": ("f16x2", False, 16, "radio_ml_conv", _mixed, False, None),
    "f16x2_batch_4096": ("f16x2", False, 16, "radio_ml_conv", None, False, "f16x2", 4096),
    "f16x2_batch_4097": ("f16x2", False, 16, "radio_ml_conv", None, False, None, 4097),
    "bf16x3_batch_4097": ("bf16x3", False, 16, "radio_ml_conv", None, False, "bf16x3", 4097),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_kernel_selection(case):
    from snn_modulation_classification_b200 import networks as N
    from snn_modulation_classification_b200 import quant
    mode, quantized, w, spec, edit, dense, want, batch = (CASES[case] + (4,))[:8]
    _pooled_spec()
    try:
        net, _ = build_pair(spec, (1, w, w), batch, K, train=False)
    finally:
        O.BUILTIN_SPECS.pop("stack16_pooled", None)
        N.BUILTIN_SPECS.pop("stack16_pooled", None)
    net.set_precision(mode)
    if quantized:
        quant.enable_quantized_weights(net)
    if edit is not None:
        edit(net)
    cells, _ = _cells(Bn=batch, Tn=6, Wn=w)
    x = cells.dense() if dense else cells
    net.reset()
    expected = _stack16_expected(net, x)
    assert net._stack16_ok(x) == expected
    # per-element time constants pass _stack16_ok; _run_stack16 then hands the window to the per-timestep kernels
    assert expected == (want is not None or case == "f16x2_per_element_tau")
    names = _kernel_names(lambda: net.test_window(x))
    stack = [k for k in names if "infer_stack16_kernel" in k]
    if want is None:
        assert not stack, stack
    else:
        assert any(STACK[want] in k for k in stack) and len(stack) == 1, sorted(names)
        assert not any("conv_mma" in k for k in names), sorted(names)


# ------------------------------------------------------------------------------------------------------------------------
# 4: refusals of the C entry point
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("edit,exc", [("mixed", NotImplementedError), ("no_w_exp", ValueError), ("a_exp", ValueError)])
def test_c_entry_refuses_mixed_forms_and_missing_exponents(edit, exc):
    from snn_modulation_classification_b200 import _lib
    net, _ = _net("f16x2", train=False)
    cells, _ = _cells(Tn=2)
    net.reset()
    layers = (_lib.ConvLayer * 3)()
    win = net._window_buffers(B)
    for i, s in enumerate(net.dcll_slices):
        s.dclllayer._fill_desc(layers[i], B, _lib.X_CELLS if i == 0 else _lib.X_DENSE, win["outs"][i])
    assert [layers[i].precision for i in range(3)] == [_lib.PREC_BF16X3, _lib.PREC_F16X2, _lib.PREC_F16X2]
    if edit == "mixed":
        layers[2].precision = _lib.PREC_BF16X3
    elif edit == "no_w_exp":
        layers[1].w_exp = None
    else:
        layers[2].a_exp = 101
    pv = [torch.empty((2 * B, 32 * 256), device="cuda") for _ in range(3)]
    pv_ptrs = (ctypes.c_void_p * 3)(*[p.data_ptr() for p in pv])
    with pytest.raises(exc, match="dcll_infer_stack16"):
        _lib.check(_lib.lib.dcll_infer_stack16(layers, 3, cells.cells[0].data_ptr(), 2, pv_ptrs, _lib.current_stream()))


# ------------------------------------------------------------------------------------------------------------------------
# 5: after training in f16x2, the stack kernel reads the moved weights and their republished exponent
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_f16x2_stack_kernel_after_learn_window():
    train_cells, _ = _cells(Tn=20, seed=4)
    y = O.to_one_hot(torch.arange(B) % K, K).cuda()
    cells, tgt = _cells()
    a, _ = _net("f16x2", 1.0, burnin=3, lr=1e-3)
    b, _ = _net("f16x2", 1.0, burnin=3, lr=1e-3)
    w0 = [s.dclllayer.i2h.weight.detach().clone() for s in a.dcll_slices]
    for n in (a, b):
        n.reset()
        n.learn_window(train_cells, y)
    for s, w in zip(a.dcll_slices, w0):
        assert (s.dclllayer.i2h.weight - w).abs().max() > 1e-3
    for sa, sb in zip(a.dcll_slices, b.dcll_slices):
        assert torch.equal(sa.dclllayer.i2h.weight, sb.dclllayer.i2h.weight)
    a.reset()
    b.reset()
    names = _kernel_names(lambda: a.test_window(cells))
    assert any(STACK["f16x2"] in k for k in names), sorted(names)
    # the exponent the kernels read is the one the library derived from the trained weights: max |w| * 2^w_exp in [2^7, 2^8)
    for s in a.dcll_slices[1:]:
        i2h = s.dclllayer.i2h
        e = int(i2h._wexp[0])
        assert 2.0 ** 7 <= float(i2h.weight.detach().abs().max()) * 2.0 ** e < 2.0 ** 8, e
    b._run_window(cells, None, False)
    _assert_stack_matches_per_step(a, b, tgt, 1.0)


# ------------------------------------------------------------------------------------------------------------------------
# 6 + 7: --precision on the CLIs
# ------------------------------------------------------------------------------------------------------------------------
def test_cli_precision_option():
    from snn_modulation_classification_b200 import test_radio_ml, train
    assert train.parse_args([]).precision == "fp32"
    assert test_radio_ml.parse_args([]).precision == "fp32"
    assert train.parse_args(["--precision", "f16x2"]).precision == "f16x2"
    with pytest.raises(SystemExit):
        train.parse_args(["--precision", "fp16"])


def _cli_args(tmp_path):
    return ["--I_resolution", "16", "--Q_resolution", "16", "--burnin", "4", "--batch_size", "8", "--batch_size_test", "8",
            "--n_test_samples", "8", "--n_iters", "12", "--n_iters_test", "12", "--radio_ml_data_dir",
            str(tmp_path / "no_such_dir"), "--synthetic", "--output", str(tmp_path / "results"), "--precision", "f16x2"]


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
def test_cli_f16x2_runs_the_stack_kernel(tmp_path):
    """--precision reaches the network in both CLIs, also after a checkpoint is restored (the precision is a mode of the
    layers that ConvNetwork takes from the parsed arguments, not a parameter)."""
    from snn_modulation_classification_b200 import test_radio_ml, train
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        fresh = {}
        names = _kernel_names(lambda: fresh.update(test_radio_ml.main(_cli_args(tmp_path), snrs=[6])))
        r = train.main(_cli_args(tmp_path) + ["--n_steps", "1", "--n_test_interval", "1"])
        ckpt = os.path.join(r["out_dir"], "parameters_0.pth")
        restored = {}
        names_r = _kernel_names(lambda: restored.update(
            test_radio_ml.main(_cli_args(tmp_path) + ["--restore_path", ckpt], snrs=[6])))
    finally:
        os.chdir(cwd)
    for ev, ks in ((fresh, names), (restored, names_r)):
        assert any(STACK["f16x2"] in k for k in ks), sorted(ks)
        assert not any("conv_mma" in k for k in ks), sorted(ks)
        assert ev["accs"].shape == (1, 3)
        assert [s.dclllayer.i2h.precision for s in ev["net"].dcll_slices] == ["f16x2"] * 3
    assert [s.dclllayer.i2h.precision for s in r["net"].dcll_slices] == ["f16x2"] * 3
    assert np.isfinite(r["acc_test"]).all()
