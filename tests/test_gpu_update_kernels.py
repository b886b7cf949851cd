"""Fused Adam updates and output-layer gradients against float64, on every dispatch branch (needs a B200: pytest -m gpu).

Protocol (one training step of one layer):
  * A runs the NON-fused route (torch.optim.SGD, lr 0): the device writes the raw gradients into .grad through the same
    reduction kernels as the fused route, with apply_update = 0;
  * B is an identical layer (same parameters, neuron state and input) that runs the FUSED route (plain torch.optim.Adam)
    with pre-seeded moments (step k, signed exp_avg scaled like |g|, positive exp_avg_sq scaled like g^2).
B's parameters, moments and step count are compared with Adam computed in float64 from A's gradients and the pre-seeded state
(the op order of torch/optim/adam.py, _single_tensor_adam), and with torch.optim.Adam(foreach=False) run in float32 on the
CPU on the same inputs.  A's gradients are compared with a float64 restatement of the local gradient, computed from the
device's own pv, read-outs and pool argmax, with a per-element bound proportional to the sum of |terms|.

Every case asserts that it reaches the kernel it is named for, through `readout_branch` / `i2h_branch` (the launchers'
selection conditions restated) and through the kernel names the CUDA profiler records.
"""
import ctypes
import math
import re
from collections import namedtuple

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as Fn

pytestmark = pytest.mark.gpu

U = 2.0 ** -24          # float32 unit roundoff
EPS32 = 2.0 ** -23      # float32 machine epsilon: an upper bound on ulp(x) / |x|
STEP0 = 5               # pre-seeded optimizer step count

# torch defaults; the training CLI's optimizer (train.py: betas (0, beta), weight_decay 10); one where every term matters
HYPERS = {
    "torch_default": dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0),
    "train_cli": dict(lr=1e-4, betas=(0.0, 0.95), eps=1e-8, weight_decay=10.0),
    "all_terms": dict(lr=1e-3, betas=(0.5, 0.9), eps=1e-3, weight_decay=1e-2),
}

Case = namedtuple("Case", "cin cout k im pool K B out prec branch")


# ------------------------------------------------------------------------------------------------------------------------
# which kernel a layer reaches: the selection conditions of launch_readout_bwd (readout.cu) and launch_wgrad (wgrad.cu)
# ------------------------------------------------------------------------------------------------------------------------
def _kmax(K):
    return 16 if K <= 16 else (24 if K <= 24 else 32)


def _aligned(n, *ts):
    return all(t is None or t.data_ptr() % n == 0 for t in ts)


def _geometry(lay):
    hc, wc = lay.i2h.get_output_shape(lay.im_dims)
    hp, wp = lay.get_output_shape()
    return hc, wc, hp, wp, lay.out_channels * hp * wp


def wgrad_tc2_supported(lay):
    """wgrad_tc2.cu: tensor-core precision on an instantiated 7x7 32->32 shape without pooling, even conv height, conv width
    a multiple of 8, K <= 32 (tensor_core_ok() is the host's restatement of tc_supported)."""
    i2h = lay.i2h
    hc, wc, _, _, _ = _geometry(lay)
    return (i2h.precision in ("bf16x3", "f16x2") and i2h.tensor_core_ok() and max(lay.pooling) == 1
            and i2h.in_channels == 32 and wc % 8 == 0 and hc % 2 == 0 and lay.target_size <= 32)


def readout_branch(lay, B, opt2=None, apply=True):
    """Kernel that computes the output_ gradient (and its Adam step) in launch_readout_bwd."""
    _, outs, _ = lay._ctx
    K = lay.target_size
    _, _, _, _, F = _geometry(lay)
    packed = F % 2 == 0 and _aligned(8, outs["pv"], lay.i2o.weight, lay._g_u)
    big_out = -(-F // 256) >= 2 * 148
    st = opt2.state.get(lay.output_.weight, {}) if opt2 is not None else {}
    packed_out = big_out and packed and _aligned(8, lay.output_.weight, st.get("exp_avg"), st.get("exp_avg_sq"),
                                                 lay.output_.weight.grad)
    fused_out = big_out and not packed_out and not wgrad_tc2_supported(lay)
    if packed_out:
        nb = B - 64 * ((B - 1) // 64)                       # rows of the last 64-row batch block
        chained = apply and K == _kmax(K) and nb // 8 >= 3  # chain_ok and >= RB2_NG - 1 full groups of UB = 8 rows
        return "wout_grad_adam2/chained" if chained else "wout_grad_adam2/plain"
    if fused_out:
        return "readout_bwd<KM,true>"
    return "wout_grad_adam<8>"


def i2h_branch(lay):
    """Kernel that applies Adam to i2h.{weight,bias}."""
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import DenseDCLLlayer
    if isinstance(lay, DenseDCLLlayer):
        return "adam_flat"
    if wgrad_tc2_supported(lay):
        return "reduce_adam_rp"
    i2h = lay.i2h
    tc = i2h.precision in ("bf16x3", "f16x2") and i2h.tensor_core_ok() and max(lay.pooling) == 1
    f16 = i2h.precision == "f16x2" and i2h.in_channels == 32
    return "wgrad_tc+reduce_adam" if tc and not f16 else "wgrad+reduce_adam"


# kernel-name patterns (demangled, spaces removed) that the profiler must show for each branch
KERNELS = {
    "wout_grad_adam2/chained": r"wout_grad_adam2_kernel<%d>",
    "wout_grad_adam2/plain": r"wout_grad_adam2_kernel<%d>",
    "wout_grad_adam<8>": r"wout_grad_adam_kernel<8>",
    "readout_bwd<KM,true>": r"readout_bwd_kernel<%d,true>",
    "reduce_adam_rp": r"reduce_adam_rp_kernel",
    "wgrad_tc+reduce_adam": r"wgrad_tc_kernel|reduce_adam_kernel",
    "wgrad+reduce_adam": r"wgrad_kernel<|reduce_adam_kernel",
    "adam_flat": r"adam_flat_kernel",
}


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key.replace(" ", "") for e in prof.key_averages()}


def _assert_ran(names, branch, K=None):
    pats = KERNELS[branch].split("|")
    for pat in pats:
        pat = pat % _kmax(K) if "%d" in pat else pat
        assert any(re.search(pat, n) for n in names), (branch, pat, sorted(n for n in names if "kernel" in n))


# ------------------------------------------------------------------------------------------------------------------------
# layers
# ------------------------------------------------------------------------------------------------------------------------
def _conv(c, seed=0):
    """Conv2dDCLLlayer on the device whose pv spreads over (0, 1) without reaching float32's subnormal range: traces after a
    step are ~tau_m tau_s (~80) per input spike, so the weights are ~0.15 / sqrt(fan-in)."""
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import Conv2dDCLLlayer
    torch.manual_seed(seed)
    lay = Conv2dDCLLlayer(c.cin, c.cout, kernel_size=c.k, im_dims=c.im, target_size=c.K, pooling=c.pool, padding=c.k // 2,
                          alpha=.92, alphas=.85, output_layer=c.out)
    g = torch.Generator().manual_seed(100 + seed)
    with torch.no_grad():
        lay.i2h.weight.copy_(torch.randn(lay.i2h.weight.shape, generator=g) * (0.15 / math.sqrt(c.cin * c.k * c.k)))
        lay.i2h.bias.copy_(torch.randn(c.cout, generator=g) * 0.5)
    lay.i2h.precision = c.prec
    return lay.cuda()


def _dense(n_in, n_out, K, seed=0):
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import DenseDCLLlayer
    torch.manual_seed(seed)
    lay = DenseDCLLlayer(n_in, n_out, target_size=K)
    g = torch.Generator().manual_seed(100 + seed)
    with torch.no_grad():
        lay.i2h.weight.copy_(torch.randn(n_out, n_in, generator=g) * (0.15 / math.sqrt(n_in)))
        lay.i2h.bias.copy_(torch.randn(n_out, generator=g) * 0.5)
    return lay.cuda()


def _slice(lay, B, optimizer, kw):
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import DCLLClassification
    return DCLLClassification(lay, batch_size=B, loss=nn.SmoothL1Loss if optimizer else None, optimizer=optimizer,
                              kwargs_optimizer=kw, burnin=0)


def _inputs(lay, B, seed):
    """(neuron state, input, one-hot target) on the device; traces in [0, 2]."""
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import DenseDCLLlayer
    g = torch.Generator().manual_seed(seed)
    if isinstance(lay, DenseDCLLlayer):
        shape = (B, lay.in_channels)
    else:
        shape = (B, lay.in_channels) + tuple(int(v) for v in lay.im_dims)
    st = (torch.rand(shape, generator=g), 2 * torch.rand(shape, generator=g))
    x = (torch.rand(shape, generator=g) < 0.1).float()
    y = torch.zeros(B, lay.target_size)
    y[torch.arange(B), torch.randint(0, lay.target_size, (B,), generator=g)] = 1.0
    return tuple(t.cuda() for t in st), x.cuda(), y.cuda()


def _set_state(lay, st):
    lay.i2h.state = lay.i2h.NeuronState(*[t.clone() for t in st])


def _params(s):
    lay = s.dclllayer
    ps = [lay.i2h.weight, lay.i2h.bias]
    return ps + ([lay.output_.weight, lay.output_.bias] if lay.output_layer else [])


def _opt_of(s, p):
    lay = s.dclllayer
    return s.optimizer2 if lay.output_layer and (p is lay.output_.weight or p is lay.output_.bias) else s.optimizer


def _pair(make, B, hp, seed=1):
    """Slices A (non-fused, SGD lr 0) and B (fused Adam with hyper-parameters hp on both optimizers), same state."""
    a = _slice(make(), B, torch.optim.SGD, {"lr": 0.0})
    b = _slice(make(), B, torch.optim.Adam, dict(hp))
    if a.dclllayer.output_layer:                      # optimizer2 is built with lr 1e-4 and otherwise default arguments
        a.optimizer2.param_groups[0]["lr"] = 0.0
        b.optimizer2.param_groups[0].update({k: v for k, v in b.optimizer.param_groups[0].items() if k != "params"})
    st, x, y = _inputs(a.dclllayer, B, seed)
    for s in (a, b):
        _set_state(s.dclllayer, st)
    return a, b, x, y


def _preseed(b, grads, hp, seed=7):
    """Adam state of every parameter of B: step STEP0, exp_avg ~ |g| N(0, 1/4), exp_avg_sq ~ g^2 [1/4, 1); returns the seeds."""
    g = torch.Generator().manual_seed(seed)
    seeds = []
    for p, gr in zip(_params(b), grads):
        s = gr.abs() + hp["weight_decay"] * p.detach().abs()
        s = (s + s.mean() + 1e-12).cpu()
        m0 = (0.5 * s * torch.randn(s.shape, generator=g)).float().cuda()
        v0 = (s * (0.5 + 0.5 * torch.rand(s.shape, generator=g))).square().float().cuda()
        _opt_of(b, p).state[p] = {"step": torch.tensor(float(STEP0)), "exp_avg": m0.clone(), "exp_avg_sq": v0.clone()}
        seeds.append((p.detach().clone(), m0, v0))
    return seeds


# ------------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------------
def _ulp32(x):
    """ulp of float32(x), elementwise (2^-149 at zero)."""
    m, e = torch.frexp(x.float())
    u = torch.ldexp(torch.ones_like(x, dtype=torch.float64), (e.to(torch.int32) - 24).clamp(min=-149).double())
    return torch.where(m == 0, 2.0 ** -149, u)


def _adam64(w, g, m, v, step_after, hp):
    """One torch.optim.Adam step (_single_tensor_adam) in float64; also the magnitude scales of the m and v updates."""
    w, g, m, v = (t.double() for t in (w, g, m, v))
    b1, b2 = hp["betas"]
    wd = hp["weight_decay"]
    ga = g.abs() + wd * w.abs()
    if wd:
        g = g + wd * w
    m1 = m + (1 - b1) * (g - m)                                   # exp_avg.lerp_(grad, 1 - beta1)
    v1 = b2 * v + (1 - b2) * g * g                                # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    bc1, bc2 = 1 - b1 ** step_after, 1 - b2 ** step_after
    w1 = w - (hp["lr"] / bc1) * m1 / (v1.sqrt() / math.sqrt(bc2) + hp["eps"])
    return w1, m1, v1, b1 * m.abs() + (1 - b1) * ga, b2 * v + (1 - b2) * ga * ga


def _torch_adam_cpu(w0, g, m0, v0, hp):
    p = nn.Parameter(w0.detach().cpu().clone())
    p.grad = g.detach().cpu().clone()
    opt = torch.optim.Adam([p], foreach=False, **hp)
    opt.state[p] = {"step": torch.tensor(float(STEP0)), "exp_avg": m0.cpu().clone(), "exp_avg_sq": v0.cpu().clone()}
    opt.step()
    st = opt.state[p]
    return p.detach(), st["exp_avg"], st["exp_avg_sq"], float(st["step"])


def _ulp_dist(a, b):
    """Distance in float32 ulps (sign-magnitude bit patterns mapped onto a line)."""
    def line(t):
        i = t.detach().float().cpu().contiguous().view(torch.int32).long()
        return torch.where(i < 0, -(i & 0x7FFFFFFF), i)
    return (line(a) - line(b)).abs()


def _check_adam(who, p, m, v, step, w0, g, m0, v0, hp):
    w1, m1, v1, sm, sv = _adam64(w0, g, m0, v0, STEP0 + 1, hp)
    assert step == STEP0 + 1, (who, "step", step)
    for name, dev, ref, tol in (("exp_avg", m, m1, 2 * EPS32 * sm), ("exp_avg_sq", v, v1, 2 * EPS32 * sv),
                                ("param", p, w1, _ulp32(w1) + 1e-6 * hp["lr"])):
        err = (dev.double() - ref).abs()
        bad = err > tol
        assert not bool(bad.any()), (who, name, int(bad.sum()), dev.numel(), float((err / tol).max()))
    # torch.optim.Adam in float32 on the CPU, same operation order (DESIGN section 8).  Not bitwise: torch's vectorised CPU
    # kernels round a few elements of the exp_avg_sq update and of the step m / denom differently, by one ulp.  The moments
    # are compared to 1 ulp.  A one-ulp difference in exp_avg_sq moves denom = sqrt(v) / sqrt(bc2) + eps by up to two ulps
    # (sqrt, division, addition), and the step m * (-step_size) / denom adds one rounding of its own on each side: the
    # parameter is compared to 4 float32 epsilons of the step plus one ulp of the result (w0 + step can cancel, and then
    # one ulp of the step is many of the result).
    tw, tm, tv, tstep = _torch_adam_cpu(w0, g, m0, v0, hp)
    assert tstep == step
    for name, dev, ref in (("exp_avg", m, tm), ("exp_avg_sq", v, tv)):
        d = _ulp_dist(dev, ref)
        assert int(d.max()) <= 1, (who, "torch float32", name, int((d > 0).sum()), dev.numel(), int(d.max()))
    tw = tw.to(p.device).double()
    err, tol = (p.double() - tw).abs(), 4 * EPS32 * (tw - w0.double()).abs() + _ulp32(tw)
    assert not bool((err > tol).any()), (who, "torch float32", "param", int((err > tol).sum()), p.numel(),
                                         float((err / tol).max()))


def _check_update(b, seeds, grads, hp):
    for i, (p, (w0, m0, v0), g) in enumerate(zip(_params(b), seeds, grads)):
        st = _opt_of(b, p).state[p]
        _check_adam("param %d" % i, p.detach(), st["exp_avg"], st["exp_avg_sq"], float(st["step"]), w0, g, m0, v0, hp)


def _close(who, dev, ref, absum, c):
    """|dev - ref| <= c 2^-24 sum|terms| (+ c 2^-149 for results in float32's subnormal range), elementwise."""
    err = (dev.double().reshape(ref.shape) - ref).abs()
    tol = c * U * absum + c * 2.0 ** -149
    bad = err > tol
    assert not bool(bad.any()), (who, int(bad.sum()), ref.numel(), float((err / tol).max()))


def _smoothl1_grad(o, y):
    B, K = y.shape
    return (o.double() - y.double()).clamp(-1.0, 1.0) / (B * K)


def _check_conv_grads(s, y):
    """A's gradients (FP32 mode) against float64 from the device's own pv, read-outs, pool argmax and traces."""
    lay = s.dclllayer
    _, outs, _ = lay._ctx
    B, K = y.shape
    hc, wc, hp, wp, F = _geometry(lay)
    cout = lay.out_channels
    pv = outs["pv"].double().reshape(B, F)
    g_o = _smoothl1_grad(outs["pvoutput"], y)
    if lay.output_layer:
        g_o2 = _smoothl1_grad(outs["output"], y)
        _close("gWout", lay.output_.weight.grad, g_o2.t() @ pv, g_o2.abs().t() @ pv, 4 * B)
        _close("gbout", lay.output_.bias.grad, g_o2.sum(0), g_o2.abs().sum(0), 4 * B)
    wo = lay.i2o.weight.double()
    sg = pv * (1 - pv)
    gu, gu_abs = (g_o @ wo) * sg, (g_o.abs() @ wo.abs()) * sg
    _close("g_u", lay._g_u, gu, gu_abs, 4 * (K + 2))
    gu, gu_abs = gu.reshape(B, cout, hp, wp), gu_abs.reshape(B, cout, hp, wp)
    if max(lay.pooling) > 1:
        # the pooled gradient lands on the argmax of its window (stored index dy * 2 + dx), zeros elsewhere
        idx = lay._pool_idx.long()
        G, Ga = (torch.zeros(B, cout, hc, wc, dtype=torch.float64, device=pv.device) for _ in range(2))
        for dy in range(2):
            for dx in range(2):
                sel = idx == dy * 2 + dx
                G[:, :, dy:2 * hp:2, dx:2 * wp:2] = torch.where(sel, gu, 0.0)
                Ga[:, :, dy:2 * hp:2, dx:2 * wp:2] = torch.where(sel, gu_abs, 0.0)
    else:
        G, Ga = gu, gu_abs
    c = 4 * max(B, K)
    _close("gb", lay.i2h.bias.grad, G.sum((0, 2, 3)), Ga.sum((0, 2, 3)), c)
    e1 = lay.i2h.state.eps1.double()              # the traces after the forward step: what the weight gradient contracts
    pad = lay.i2h.padding
    gw = Fn.conv2d(e1.transpose(0, 1), G.transpose(0, 1), padding=pad).transpose(0, 1)
    gw_abs = Fn.conv2d(e1.abs().transpose(0, 1), Ga.transpose(0, 1), padding=pad).transpose(0, 1)
    _close("gW", lay.i2h.weight.grad, gw, gw_abs, c)


def _check_dense_grads(s, y):
    lay = s.dclllayer
    (_, _, _, _, _), outs = lay._ctx
    B, K = y.shape
    pv = outs["pv"].double()
    g_o = _smoothl1_grad(outs["pvoutput"], y)
    wo = lay.i2o.weight.double()
    sg = pv * (1 - pv)
    gu, gu_abs = (g_o @ wo) * sg, (g_o.abs() @ wo.abs()) * sg
    e1 = lay.i2h.state.eps1.double()
    c = 4 * (B + K)
    _close("gb", lay.i2h.bias.grad, gu.sum(0), gu_abs.sum(0), c)
    _close("gW", lay.i2h.weight.grad, gu.t() @ e1, gu_abs.t() @ e1.abs(), c)


def _run_protocol(make, B, hp, check_grads):
    a, b, x, y = _pair(make, B, hp)
    a.train_dcll(x, y, regularize=False)
    grads = [p.grad.detach().clone() for p in _params(a)]
    if check_grads:
        check_grads(a, y)
    seeds = _preseed(b, grads, hp)
    names = _kernel_names(lambda: b.train_dcll(x, y, regularize=False))
    _check_update(b, seeds, grads, hp)
    return a, b, names


# ------------------------------------------------------------------------------------------------------------------------
# 1 + 2: output layer, every branch of launch_readout_bwd (FP32 mode: the forward is exact to ~1e-6)
# ------------------------------------------------------------------------------------------------------------------------
OUT_CASES = {
    # Cout 32, 49x49 conv, no pool: F = 76 832, ceil(F / 256) = 301 >= 296, even -> wout_grad_adam2
    "chained_b30_k24": Case(1, 32, 7, (49, 49), None, 24, 30, True, "fp32", "wout_grad_adam2/chained"),    # 6 rows after the ring groups
    "chained_b88_k24": Case(1, 32, 7, (49, 49), None, 24, 88, True, "fp32", "wout_grad_adam2/chained"),    # 2nd block chained
    "chained_b24_k16": Case(1, 32, 7, (49, 49), None, 16, 24, True, "fp32", "wout_grad_adam2/chained"),    # KMAX 16, TG 4
    "chained_b43_k32": Case(1, 32, 7, (49, 49), None, 32, 43, True, "fp32", "wout_grad_adam2/chained"),    # KMAX 32, TG 8
    "plain_b5_k10": Case(1, 32, 7, (49, 49), None, 10, 5, True, "fp32", "wout_grad_adam2/plain"),          # K < KMAX
    "plain_b16_k24": Case(1, 32, 7, (49, 49), None, 24, 16, True, "fp32", "wout_grad_adam2/plain"),        # 2 groups: no chain
    "plain_b70_k20": Case(1, 32, 7, (49, 49), None, 20, 70, True, "fp32", "wout_grad_adam2/plain"),        # after a full block
    # pooled 15x13 conv -> 7x6 planes, F = 336: small F; K = 17 leaves a partial group of KG = 8 outputs
    "small_b70_k17_pool": Case(2, 8, 3, (15, 13), 2, 17, 70, True, "fp32", "wout_grad_adam<8>"),
    # Cout 9, 93x93 conv: F = 77 841, odd -> the fused scalar sweep
    "fused_odd_b3_k10": Case(1, 9, 3, (93, 93), None, 10, 3, True, "fp32", "readout_bwd<KM,true>"),
    "fused_odd_b70_k10": Case(1, 9, 3, (93, 93), None, 10, 70, True, "fp32", "readout_bwd<KM,true>"),
}


@pytest.mark.parametrize("hyper", sorted(HYPERS))
@pytest.mark.parametrize("case", sorted(OUT_CASES))
def test_output_layer_gradients_and_adam(case, hyper):
    c, hp = OUT_CASES[case], HYPERS[hyper]
    a, b, names = _run_protocol(lambda: _conv(c), c.B, hp, _check_conv_grads)
    assert readout_branch(a.dclllayer, c.B, a.optimizer2, apply=False) == c.branch.replace("chained", "plain")
    assert readout_branch(b.dclllayer, c.B, b.optimizer2) == c.branch
    _assert_ran(names, c.branch, c.K)
    assert i2h_branch(b.dclllayer) == "wgrad+reduce_adam"


# ------------------------------------------------------------------------------------------------------------------------
# 3: i2h Adam paths
# ------------------------------------------------------------------------------------------------------------------------
I2H_CASES = {
    "fp32_7x7": Case(2, 8, 7, (20, 20), None, 10, 4, False, "fp32", "wgrad+reduce_adam"),
    "tc_layer0_bf16x3": Case(1, 32, 7, (16, 16), None, 24, 4, False, "bf16x3", "wgrad_tc+reduce_adam"),
    "rowpair_bf16x3": Case(32, 32, 7, (16, 16), None, 24, 4, False, "bf16x3", "reduce_adam_rp"),
    "rowpair_f16x2": Case(32, 32, 7, (16, 16), None, 24, 4, False, "f16x2", "reduce_adam_rp"),
}
# (B, In, Out, K) around the 32 x 32 tile of dense.cu's SGEMM
DENSE_CASES = [(1, 1, 1, 1), (33, 70, 129, 10), (64, 257, 32, 32)]


@pytest.mark.parametrize("hyper", sorted(HYPERS))
@pytest.mark.parametrize("case", sorted(I2H_CASES))
def test_i2h_conv_adam(case, hyper):
    c = I2H_CASES[case]
    _, b, names = _run_protocol(lambda: _conv(c), c.B, HYPERS[hyper], _check_conv_grads if c.prec == "fp32" else None)
    assert i2h_branch(b.dclllayer) == c.branch
    assert b.dclllayer.i2h.tensor_core_ok() == (c.prec != "fp32")
    _assert_ran(names, c.branch)


@pytest.mark.parametrize("hyper", sorted(HYPERS))
@pytest.mark.parametrize("B,n_in,n_out,K", DENSE_CASES)
def test_dense_adam(B, n_in, n_out, K, hyper):
    _, b, names = _run_protocol(lambda: _dense(n_in, n_out, K), B, HYPERS[hyper], _check_dense_grads)
    assert i2h_branch(b.dclllayer) == "adam_flat"
    _assert_ran(names, "adam_flat")


@pytest.mark.parametrize("hyper", sorted(HYPERS))
def test_conv_apply_update(hyper):
    """dcll_conv_apply_update (Adam on externally reduced gradients, then the kernel-side weight copies) through the C ABI
    with a hand-filled TrainArgs: parameters and moments against float64, and the next forward sees the new weights."""
    from snn_modulation_classification_b200 import _lib
    hp = HYPERS[hyper]
    c = Case(2, 8, 3, (12, 12), None, 10, 4, True, "fp32", None)
    lay = _conv(c)
    lay.init_hiddens(c.B)
    st, x, _ = _inputs(lay, c.B, seed=3)
    _set_state(lay, st)
    desc = _lib.ConvLayer()
    lay._fill_desc(desc, c.B, _lib.X_DENSE, None)
    g = torch.Generator().manual_seed(4)
    params = [lay.i2h.weight, lay.i2h.bias, lay.output_.weight, lay.output_.bias]
    grads = [(torch.randn(p.shape, generator=g) * 1e-3).cuda() for p in params]
    seeds = []
    for p, gr in zip(params, grads):
        s = (gr.abs() + hp["weight_decay"] * p.detach().abs()).cpu() + 1e-4
        seeds.append((p.detach().clone(), (0.5 * s * torch.randn(s.shape, generator=g)).cuda(),
                      (s * (0.5 + 0.5 * torch.rand(s.shape, generator=g))).square().cuda()))
    moments = [(m0.clone(), v0.clone()) for _, m0, v0 in seeds]
    args = _lib.TrainArgs()
    args.grad_w, args.grad_b, args.grad_wout, args.grad_bout = (_lib.ptr(t) for t in grads)
    for adam, (mw, vw), (mb, vb) in ((args.adam_i2h, moments[0], moments[1]), (args.adam_out, moments[2], moments[3])):
        adam.lr, adam.beta1, adam.beta2 = hp["lr"], hp["betas"][0], hp["betas"][1]
        adam.eps, adam.weight_decay, adam.step = hp["eps"], hp["weight_decay"], STEP0
        adam.m_w, adam.v_w, adam.m_b, adam.v_b = _lib.ptr(mw), _lib.ptr(vw), _lib.ptr(mb), _lib.ptr(vb)
    _lib.check(_lib.lib.dcll_conv_apply_update(ctypes.byref(desc), ctypes.byref(args), _lib.current_stream()))
    torch.cuda.synchronize()
    assert args.adam_i2h.step == STEP0 + 1 and args.adam_out.step == STEP0 + 1
    for i, (p, (w0, m0, v0), gr, (m, v)) in enumerate(zip(params, seeds, grads, moments)):
        _check_adam("param %d" % i, p.detach(), m, v, float(STEP0 + 1), w0, gr, m0, v0, hp)
    # the weights changed behind Python's back (no parameter version bump): only the library's own sync refreshes weight_t
    _set_state(lay, st)
    got = lay.forward(x)
    fresh = _conv(c, seed=9)
    fresh.load_state_dict(lay.state_dict())
    fresh.init_hiddens(c.B)
    _set_state(fresh, st)
    want = fresh.forward(x)
    for u, w in zip(got, want):
        assert torch.equal(u, w)


# ------------------------------------------------------------------------------------------------------------------------
# 4: the kernel-side weight images follow the update
# ------------------------------------------------------------------------------------------------------------------------
IMAGE_CASES = {
    "fp32": (I2H_CASES["fp32_7x7"], 1e-3),
    "bf16x3_layer0": (I2H_CASES["tc_layer0_bf16x3"], 1e-3),
    "bf16x3_rowpair": (I2H_CASES["rowpair_bf16x3"], 1e-3),
    # lr far below max|w| ~ 0.1: the fp16 image's exponent (from the binade of max|w|) cannot change in one step
    "f16x2_rowpair": (I2H_CASES["rowpair_f16x2"], 1e-6),
}


def _max_binade(w):
    return math.frexp(float(w.detach().abs().max()))[1]


def _next_forward(s, st, x):
    _set_state(s.dclllayer, st)
    s.forward(x, ignore_burnin=True)
    _, outs, _ = s.dclllayer._ctx
    return [outs[k].clone() for k in ("pvmem", "pvoutput", "spikes")]


@pytest.mark.parametrize("route", ["fused_adam", "amsgrad"])
@pytest.mark.parametrize("case", sorted(IMAGE_CASES))
def test_next_forward_sees_updated_weights(case, route):
    """After one training step, the next forward of the trained layer equals bit for bit the forward of a fresh layer that
    received the same parameters through load_state_dict (dcll_conv_sync_weights): weight_t, the bf16 {hi,lo} image and the
    fp16 image with its exponent were refreshed by the update.  Route 'amsgrad' is not plain Adam: the gradient goes to
    .grad and torch's optimizer.step() changes the parameter, which the next forward must notice by its version."""
    c, lr = IMAGE_CASES[case]
    kw = {"lr": lr, "betas": (0.9, 0.999), "amsgrad": route == "amsgrad"}
    b = _slice(_conv(c), c.B, torch.optim.Adam, kw)
    st, x, y = _inputs(b.dclllayer, c.B, seed=1)
    st2, x2, _ = _inputs(b.dclllayer, c.B, seed=2)
    before = _next_forward(_slice(_conv(c), c.B, None, {}), st2, x2)
    w_before = b.dclllayer.i2h.weight.detach().clone()
    _set_state(b.dclllayer, st)
    b.train_dcll(x, y, regularize=False)
    lay = b.dclllayer
    assert float((lay.i2h.weight.detach() - w_before).abs().max()) > 0
    if c.prec == "f16x2":
        assert _max_binade(lay.i2h.weight) == _max_binade(w_before)
        assert lay._ctx[0].precision == 2                                 # PREC_F16X2
    got = _next_forward(b, st2, x2)
    fresh = _slice(_conv(c, seed=9), c.B, None, {})
    fresh.load_state_dict(b.state_dict())
    want = _next_forward(fresh, st2, x2)
    for name, u, w in zip(("pvmem", "pvoutput", "spikes"), got, want):
        assert torch.equal(u, w), (name, float((u - w).abs().max()))
    assert not torch.equal(got[0], before[0])                             # the update is visible in the membrane
