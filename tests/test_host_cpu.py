"""Host-side logic and C-ABI surface, no GPU needed (no compute call is made)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from golden_util import NetFixture

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from snn_modulation_classification_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dcll_b200.h")).read()
    declared = set(re.findall(r"\b(dcll_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    assert declared == set(_lib.EXPORTS)
    so = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(so, name), name
    assert _lib.lib.dcll_abi_version() == _lib.ABI_VERSION
    assert _lib.lib.dcll_sizeof_conv_layer() == ctypes.sizeof(_lib.ConvLayer)
    assert _lib.lib.dcll_sizeof_train_args() == ctypes.sizeof(_lib.TrainArgs)


def test_argument_errors_are_reported_without_a_gpu():
    from snn_modulation_classification_b200 import _lib
    with pytest.raises(ValueError, match="null pointer"):
        _lib.check(_lib.lib.dcll_iq_encode(None, 4, 8, -1.0, 1.0, -1.0, 1.0, 16, 16, 0, 8, 1, None, None))
    with pytest.raises(ValueError, match="exceeds"):
        _lib.check(_lib.lib.dcll_iq_encode(1024, 4, 8, -1.0, 1.0, -1.0, 1.0, 16, 16, 4, 8, 1, 2048, None))
    d = _lib.ConvLayer()
    d.B, d.Cin, d.H, d.W, d.Cout, d.KH, d.KW, d.padH, d.padW, d.poolH, d.poolW, d.K = 4, 1, 16, 16, 32, 7, 7, 3, 3, 1, 1, 24
    assert _lib.lib.dcll_conv_workspace_bytes(ctypes.byref(d)) > 0
    with pytest.raises(ValueError):
        _lib.check(_lib.lib.dcll_conv_step_fwd(ctypes.byref(d), None, None, None))
    d.poolH = 3
    with pytest.raises(NotImplementedError):
        _lib.check(_lib.lib.dcll_conv_step_fwd(ctypes.byref(d), 1024, None, None))


@pytest.fixture
def cpu_modules(monkeypatch):
    """Construction-only use of the host mirror on CPU (kernels are never called)."""
    from snn_modulation_classification_b200 import networks as N
    from snn_modulation_classification_b200.dcll import pytorch_libdcll as L
    monkeypatch.setattr(L, "device", "cpu")
    monkeypatch.setattr(N, "device", "cpu")
    return L, N


def _build(N, spec, im_dims, B, K, arp, seed=1, train=True):
    from util_build import make_args
    torch.manual_seed(seed)
    np.random.seed(seed)
    kw = dict(loss=torch.nn.SmoothL1Loss, opt=torch.optim.Adam, opt_param={"betas": [0.0, 0.95], "weight_decay": 10.0},
              learning_rates=[1e-6]) if train else dict(loss=None, opt=None, opt_param={}, learning_rates=None)
    return N.ConvNetwork(make_args(arp), im_dims, B, N.load_network_spec(spec), K, act=torch.nn.Sigmoid(), burnin=50, **kw)


@pytest.mark.parametrize("name", ["radio8_train", "radio8_arp_infer", "mnist_train", "radioref_train"])
def test_state_dict_keys_and_shapes_match_reference_fixture(cpu_modules, name):
    L, N = cpu_modules
    fx = NetFixture(name)
    net = _build(N, fx.spec_name, fx.im_dims, fx.B, fx.K, fx.arp, train=fx.train)
    sd = net.state_dict()
    assert set(sd.keys()) == set(fx.state_dict.keys())
    for k, v in fx.state_dict.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    net.load_state_dict(fx.state_dict, strict=True)


@pytest.mark.parametrize("name", ["radio8_train", "radio8_arp_train", "mnist_train", "radioref_train"])
def test_constructors_consume_rng_like_the_reference(cpu_modules, name):
    """Same seeds -> bit-identical initial parameters and time constants (torch + numpy RNG order:
    reset_parameters -> nn.Linear inits -> reset_lc_parameters -> randomize_tau: tau_m then tau_s).  The fixture holds the
    state_dict of the reference's own ConvNetwork built at seed 1 (tests/golden/make_golden.py)."""
    L, N = cpu_modules
    fx = NetFixture(name)
    net = _build(N, fx.spec_name, fx.im_dims, fx.B, fx.K, fx.arp)
    net.reset(True)
    a, b = fx.state_dict, net.state_dict()
    assert list(a.keys()) == list(b.keys())
    for k in a:
        assert torch.equal(a[k], b[k]), k
    # the reference's optimizer groups (train.py:224-225 touches them)
    for s in net.dcll_slices:
        assert s.optimizer.param_groups[-1]["lr"] == 1e-6 and s.optimizer.param_groups[-1]["weight_decay"] == 10.0
    assert net.dcll_slices[-1].optimizer2.param_groups[-1]["lr"] == 1e-4
    assert not hasattr(net.dcll_slices[0], "optimizer2")


def test_load_network_spec_schema(tmp_path, cpu_modules):
    L, N = cpu_modules
    p = tmp_path / "net.yaml"
    p.write_text('conv_layers:\n  - out_channels: 8\n    kernel_size: "(1, 3)"\n    padding: "(0, 1)"\n    pooling: 2\n')
    convs = N.load_network_spec(str(p))
    assert convs == [dict(out_channels=8, kernel_size=(1, 3), padding=(0, 1), pooling=2)]
    assert N.load_network_spec("networks/radio_ml_conv_ref.yaml")[0]["kernel_size"] == (1, 3)
    assert len(N.load_network_spec("networks/mnist_conv.yaml")) == 3
    with pytest.raises(FileNotFoundError):
        N.load_network_spec("networks/nope.yaml")


def test_layer_constructor_errors(cpu_modules):
    L, N = cpu_modules
    with pytest.raises(ValueError):
        L.ContinuousConv2D(3, 8, 7, groups=2)                       # ref :316-319
    with pytest.raises(Exception, match="Non-spiking"):
        L.Conv2dDCLLlayer(1, 8, wrp=1.0, spiking=False)             # ref :556-558
    lay = L.Conv2dDCLLlayer(1, 16, kernel_size=7, padding=2, pooling=2, im_dims=(28, 28), target_size=10,
                            output_layer=True)
    assert lay.get_flat_size() == 16 * 13 * 13 and tuple(lay.output_shape) == (13, 13)
    assert lay.i2o.weight.shape == (10, 2704) and not lay.i2o.weight.requires_grad
    assert lay.output_.weight.requires_grad
    lay.init_hiddens(3)
    assert lay.i2h.state.eps0.shape == (3, 1, 28, 28) and lay.i2h.alpha.shape == (1,)
    with pytest.raises(RuntimeError, match="no CPU path"):
        lay.forward(torch.zeros(3, 1, 28, 28))                      # product path fails loudly without CUDA


def test_device_clout_counting_rule_is_host_side(cpu_modules):
    L, N = cpu_modules
    c = L.DeviceClout()
    assert len(c) == 0 and np.array(c).shape[0] == 0


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import importlib
    from snn_modulation_classification_b200 import _lib
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libdcll_b200.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib._load()


def test_every_kernel_waits_for_its_predecessor_and_every_launch_is_chained():
    """Programmatic dependent launch (DESIGN 4.6) is only safe if EVERY kernel executes griddepcontrol.wait before touching
    global memory and every launch goes through launch_k: a static check over the CUDA sources."""
    import glob
    import re
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "snn_modulation_classification_b200", "csrc")
    n_kernels = 0
    for path in sorted(glob.glob(os.path.join(csrc, "*.cu"))):
        src = open(path).read()
        assert "<<<" not in src, "%s launches a kernel without launch_k" % os.path.basename(path)
        for m in re.finditer(r"__global__", src):
            # body = from the first '{' after the parameter list to the matching '}'
            i = src.index("(", m.end())
            depth, j = 0, i
            while True:                                   # skip __launch_bounds__(...) and the parameter list
                if src[j] == "(":
                    depth += 1
                elif src[j] == ")":
                    depth -= 1
                    if depth == 0 and src[j + 1:].lstrip().startswith("{"):
                        break
                j += 1
            b0 = src.index("{", j)
            depth, k = 0, b0
            while True:
                if src[k] == "{":
                    depth += 1
                elif src[k] == "}":
                    depth -= 1
                    if depth == 0:
                        break
                k += 1
            body = src[b0:k]
            assert "pdl_entry();" in body, "kernel near %s:%d has no pdl_entry()" % (os.path.basename(path), src[:m.start()].count("\n") + 1)
            n_kernels += 1
    assert n_kernels >= 30


def test_f16x2_host_side_exponents_and_layer_selection(cpu_modules):
    """'f16x2' host logic (no GPU): which layers get the fp16 form, and the power-of-two exponents the host derives --
    trace image: 2^a_exp * tau_s/(1-alphas) * tau_m/(1-alpha) <= 2^15 (fp16 maximum 65504) and within a factor 2 of it;
    gradient image: 2^g_exp * 16 * max|Wo| / (4 B) <= 2^14."""
    import math
    import types
    import numpy as np
    import torch
    L, _ = cpu_modules
    np.random.seed(0)
    torch.manual_seed(0)
    core = L.ContinuousConv2D(32, 32, kernel_size=7, padding=3, random_tau=False)
    core.precision = "f16x2"
    assert core.tensor_core_ok() and core.f16_ok(128, 128) and core.f16_ok(16, 16) and core.f16_ok(40, 24)
    assert not core.f16_ok(21, 45) and not core.f16_ok(16, 20)            # odd conv height / conv width not a multiple of 8
    first = L.ContinuousConv2D(1, 32, kernel_size=7, padding=3, random_tau=False)
    first.precision = "f16x2"
    assert first.tensor_core_ok() and not first.f16_ok(128, 128)          # one input channel keeps the split-bf16 kernels
    a_exp = core._trace_exp()
    bound = float(core.tau_s__dt / (1 - core.alphas) * core.tau_m__dt / (1 - core.alpha))
    assert bound * 2.0 ** a_exp <= 32768.0 < bound * 2.0 ** (a_exp + 1)
    lay = types.SimpleNamespace(i2o=torch.nn.Linear(8, 4))
    g_exp = L.Conv2dDCLLlayer._grad_exp(lay, 64)
    gb = float(lay.i2o.weight.detach().abs().max()) / (4 * 64) * 16
    assert gb * 2.0 ** g_exp <= 16384.0 < gb * 2.0 ** (g_exp + 1)
    assert L.Conv2dDCLLlayer._grad_exp(lay, 64) == g_exp                   # cached per (weight version, batch)
    assert math.isfinite(a_exp) and math.isfinite(g_exp)
