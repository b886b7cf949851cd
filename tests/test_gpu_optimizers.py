"""AdamW, Adamax, NAdam and RAdam applied on the device (train.py --optim_type), against float64 and torch.

The first test needs no GPU.  The GPU tests reuse the protocol of test_gpu_update_kernels.py: layer A takes the non-fused
route (SGD, lr 0) and leaves the raw gradients in .grad; the identical layer B takes the fused route with the rule under test
and pre-seeded state.  B's parameters and state are compared with that rule computed in float64 from A's gradients (the
operation order of torch's _single_tensor_<rule>), and with torch.optim.<Class>(foreach=False) in float32 on the CPU.
"""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from test_gpu_update_kernels import (DENSE_CASES, EPS32, I2H_CASES, IMAGE_CASES, OUT_CASES, Case, _conv, _dense,
                                     _inputs, _kernel_names, _kmax, _next_forward, _opt_of, _params, _set_state, _slice,
                                     _ulp32, _ulp_dist, i2h_branch, readout_branch)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RULES = {"AdamW": torch.optim.AdamW, "Adamax": torch.optim.Adamax, "NAdam": torch.optim.NAdam, "RAdam": torch.optim.RAdam}
CLI = dict(lr=1e-4, betas=(0.0, 0.95), weight_decay=10.0)            # train.py: betas (0, beta), weight_decay 10
# (hyper-parameters, pre-seeded step count): the class defaults, the CLI's, and NAdam / RAdam with decoupled weight decay, at
# step 6, where RAdam's rho_t is 5.99 (beta2 0.999) or 5.70 (beta2 0.95): rectified.  RAdam also runs at step 1, where
# rho_t = 1 <= 5: not rectified.
HYPERS = {"default": ({}, 5), "cli": (CLI, 5), "decoupled": (dict(CLI, decoupled_weight_decay=True), 5), "step1": ({}, 0)}
RULE_HYPERS = {"AdamW": ["default", "cli"], "Adamax": ["default", "cli"], "NAdam": ["default", "cli", "decoupled"],
               "RAdam": ["default", "cli", "decoupled", "step1"]}
CASES = [(r, h) for r in sorted(RULES) for h in RULE_HYPERS[r]]


# ------------------------------------------------------------------------------------------------------------------------
# 1: which optimizers the device applies (no GPU)
# ------------------------------------------------------------------------------------------------------------------------
def test_device_optim_classifier():
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import _device_optim, _is_plain_adam
    p = [nn.Parameter(torch.zeros(3))]
    O = torch.optim
    assert _device_optim(O.AdamW(p)) == _lib.OPT_ADAMW
    assert _device_optim(O.Adam(p, decoupled_weight_decay=True)) == _lib.OPT_ADAMW
    assert _device_optim(O.Adamax(p, betas=[0, 0.95], weight_decay=10)) == _lib.OPT_ADAMAX
    assert _device_optim(O.NAdam(p)) == _device_optim(O.NAdam(p, decoupled_weight_decay=True)) == _lib.OPT_NADAM
    assert _device_optim(O.RAdam(p)) == _device_optim(O.RAdam(p, decoupled_weight_decay=True)) == _lib.OPT_RADAM
    assert _device_optim(O.AdamW(p, foreach=True)) == _lib.OPT_ADAMW          # foreach / fused are ignored

    class MyNAdam(O.NAdam):
        pass
    two = O.RAdam([{"params": p}, {"params": [nn.Parameter(torch.zeros(1))]}])
    for opt in (O.SGD(p, lr=0.1), O.Adam(p), O.AdamW(p, amsgrad=True), O.Adam(p, amsgrad=True, decoupled_weight_decay=True),
                O.NAdam(p, maximize=True), O.RAdam(p, capturable=True), O.Adamax(p, differentiable=True),
                O.AdamW(p, lr=torch.tensor(1e-3)), two, MyNAdam(p)):
        assert _device_optim(opt) is None, opt
    assert _is_plain_adam(O.Adam(p)) and not _is_plain_adam(O.AdamW(p))


# ------------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------------
def _group(opt):
    g = dict(opt.param_groups[0])
    g.pop("params")
    return g


def _kwargs(opt, **over):
    """Constructor arguments of type(opt) that rebuild its hyper-parameters."""
    import inspect
    names = inspect.signature(type(opt).__init__).parameters
    return dict({k: v for k, v in _group(opt).items() if k in names}, **over)


def _mu(b1, md, t):
    return b1 * (1.0 - 0.5 * 0.96 ** (t * md))


def _mu_product(b1, md, steps):
    """torch's float32 state['mu_product'] after `steps` NAdam steps (a float32 tensor times a python float)."""
    mp = torch.tensor(1.0)
    for t in range(1, steps + 1):
        mp *= _mu(b1, md, t)
    return mp


def _rule64(name, g, w, gr, m, v, t, mp):
    """One step of rule `name` with hyper-parameters g in float64, the op order of torch's _single_tensor_<rule>.  mp: NAdam's
    float32 mu_product before the step.  Returns (w1, m1, v1, magnitude scales of m1 and v1, and the magnitude scale of
    w1 - w: the sum of |terms|, with exp_avg's scale in place of |exp_avg|, which can cancel)."""
    w, gr, m, v = (x.double() for x in (w, gr, m, v))
    lr, (b1, b2), eps, wd = g["lr"], g["betas"], g["eps"], g["weight_decay"]
    decoupled = name == "AdamW" or g.get("decoupled_weight_decay", False)
    terms = torch.zeros_like(w)
    ga = gr.abs()
    if wd and decoupled:
        terms = terms + (lr * wd * w).abs()
        w = w * (1 - lr * wd)
    elif wd:
        ga = ga + wd * w.abs()
        gr = gr + wd * w
    m1 = m + (1 - b1) * (gr - m)
    sm = b1 * m.abs() + (1 - b1) * ga
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    if name == "Adamax":
        v1 = torch.maximum(b2 * v, gr.abs() + eps)
        d = (lr / bc1) * m1 / v1
        return w - d, m1, v1, sm, v1, terms + (lr / bc1) * sm / v1
    v1 = b2 * v + (1 - b2) * gr * gr
    sv = b2 * v + (1 - b2) * ga * ga
    if name == "AdamW":
        denom = v1.sqrt() / math.sqrt(bc2) + eps
        d = (lr / bc1) * m1 / denom
        return w - d, m1, v1, sm, sv, terms + (lr / bc1) * sm / denom
    if name == "NAdam":
        md = g["momentum_decay"]
        mu, mu_next = _mu(b1, md, t), _mu(b1, md, t + 1)
        mp = float(torch.tensor(mp) * mu)
        denom = (v1 / bc2).sqrt() + eps
        c1, c2 = lr * (1 - mu) / (1 - mp), lr * mu_next / (1 - mp * mu_next)
        d1, d2 = c1 * gr / denom, c2 * m1 / denom
        return w - d1 - d2, m1, v1, sm, sv, terms + (c1 * ga + c2 * sm) / denom
    rho_inf = 2 / (1 - b2) - 1
    rho_t = rho_inf - 2 * t * b2 ** t / bc2
    f = lr / bc1
    if rho_t > 5:
        rect = math.sqrt((rho_t - 4) * (rho_t - 2) * rho_inf / ((rho_inf - 4) * (rho_inf - 2) * rho_t))
        f = f * math.sqrt(bc2) / (v1.sqrt() + eps) * rect
    return w - m1 * f, m1, v1, sm, sv, terms + sm * f


def _vkey(name):
    return "exp_inf" if name == "Adamax" else "exp_avg_sq"


def _seed_state(name, opt, p, gr, step0, gen):
    """State of p at step `step0`: signed exp_avg ~ |g|, positive second moment / infinity norm ~ g^2 / |g|."""
    g = _group(opt)
    s = gr.abs() + g["weight_decay"] * p.detach().abs()
    s = (s + s.mean() + 1e-12).cpu()
    m0 = (0.5 * s * torch.randn(s.shape, generator=gen)).float().cuda()
    v0 = s * (0.5 + 0.5 * torch.rand(s.shape, generator=gen))
    v0 = (v0 if name == "Adamax" else v0.square()).float().cuda()
    st = {"step": torch.tensor(float(step0)), "exp_avg": m0.clone(), _vkey(name): v0.clone()}
    if name == "NAdam":
        st["mu_product"] = _mu_product(g["betas"][0], g["momentum_decay"], step0)
    opt.state[p] = st
    return p.detach().clone(), m0, v0, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in st.items()}


def _torch_cpu(name, opt, w0, gr, st0):
    p = nn.Parameter(w0.detach().cpu().clone())
    p.grad = gr.detach().cpu().clone()
    o = RULES[name]([p], **_kwargs(opt, foreach=False))
    o.state[p] = {k: v.detach().cpu().clone() for k, v in st0.items()}
    o.step()
    return p.detach(), o.state[p]


def _check_rule(who, name, opt, p, st, w0, gr, m0, v0, st0):
    """Device result against float64 and against torch in float32 on the CPU.
    Bounds, from the Adam harness (test_gpu_update_kernels.py): moments within 2 float32 epsilons of their update's
    magnitude; step count exact.  The parameter bound is widened: the Adam harness bounds the step by 1e-6 lr, since
    |m / denom| stays near 1 there, but Adamax's lr m / v and RAdam's unrectified lr m / bc1 are not bounded by lr; so the
    parameter is held to 8 epsilons of the magnitude scale of its update (the sum of |terms|, with exp_avg's scale for
    exp_avg: an exp_avg that cancels carries the absolute error of its scale) plus 2 ulps of the result (NAdam rounds the
    parameter between its two addcdivs, AdamW / decoupled decay between the decay and the step)."""
    g = _group(opt)
    step0 = float(st0["step"])
    t = step0 + 1
    mp = float(st0["mu_product"]) if name == "NAdam" else 1.0
    w1, m1, v1, sm, sv, terms = _rule64(name, g, w0, gr, m0, v0, t, mp)
    assert float(st["step"]) == t, (who, "step")
    if name == "NAdam":
        assert torch.equal(st["mu_product"], _mu_product(g["betas"][0], g["momentum_decay"], int(t))), (who, "mu_product")
    m, v = st["exp_avg"], st[_vkey(name)]
    for what, dev, ref, tol in (("exp_avg", m, m1, 2 * EPS32 * sm), (_vkey(name), v, v1, 2 * EPS32 * sv),
                                ("param", p, w1, 2 * _ulp32(w1) + 8 * EPS32 * terms)):
        err = (dev.double() - ref).abs()
        bad = err > tol
        assert not bool(bad.any()), (who, what, int(bad.sum()), dev.numel(), float((err / tol).max()))
    # torch in float32 on the CPU: moments within one ulp (its vectorised kernels round a few elements differently); the
    # parameter within the float64 bound above -- one ulp of exp_avg_sq moves each term of the update by a few epsilons, and
    # NAdam's two addcdiv terms can cancel, so the bound follows the magnitude scale of the terms, not the net step
    tw, tst = _torch_cpu(name, opt, w0, gr, st0)
    assert float(tst["step"]) == t
    for what in ("exp_avg", _vkey(name)):
        d = _ulp_dist(st[what], tst[what])
        assert int(d.max()) <= 1, (who, "torch float32", what, int((d > 0).sum()), int(d.max()))
    if name == "NAdam":
        assert torch.equal(st["mu_product"], tst["mu_product"])
    tw = tw.to(p.device).double()
    err, tol = (p.double() - tw).abs(), 8 * EPS32 * terms + 2 * _ulp32(tw)
    assert not bool((err > tol).any()), (who, "torch float32", "param", int((err > tol).sum()), float((err / tol).max()))


# the _opt kernel each branch must reach, and the Adam kernel it must not
OPT_KERNELS = {
    "wout_grad_adam2/chained": (r"wout_grad_opt2_kernel<%d>", r"wout_grad_adam2_kernel<"),
    "wout_grad_adam2/plain": (r"wout_grad_opt2_kernel<%d>", r"wout_grad_adam2_kernel<"),
    "wout_grad_adam<8>": (r"wout_grad_opt_kernel<8>", r"wout_grad_adam_kernel<"),
    "readout_bwd<KM,true>": (r"readout_bwd_opt_kernel<%d,true>", r"readout_bwd_kernel<\d+,true>"),
    "reduce_adam_rp": (r"reduce_opt_rp_kernel", r"reduce_adam_rp_kernel"),
    "wgrad_tc+reduce_adam": (r"reduce_opt_kernel", r"reduce_adam_kernel"),
    "wgrad+reduce_adam": (r"reduce_opt_kernel", r"reduce_adam_kernel"),
    "adam_flat": (r"opt_flat_kernel", r"adam_flat_kernel"),
}


def _assert_opt_ran(names, branch, K=None):
    ran, not_ran = OPT_KERNELS[branch]
    ran = ran % _kmax(K) if "%d" in ran else ran
    assert any(re.search(ran, n) for n in names), (branch, ran, sorted(n for n in names if "kernel" in n))
    assert not any(re.search(not_ran, n) for n in names), (branch, not_ran)


def _run(make, B, name, hyper):
    hp, step0 = HYPERS[hyper]
    a = _slice(make(), B, torch.optim.SGD, {"lr": 0.0})
    b = _slice(make(), B, RULES[name], dict(hp))
    if a.dclllayer.output_layer:                      # optimizer2 is built with lr 1e-4 and otherwise default arguments
        a.optimizer2.param_groups[0]["lr"] = 0.0
        b.optimizer2.param_groups[0].update({k: v for k, v in b.optimizer.param_groups[0].items() if k != "params"})
    st, x, y = _inputs(a.dclllayer, B, 1)
    for s in (a, b):
        _set_state(s.dclllayer, st)
    a.train_dcll(x, y, regularize=False)
    grads = [p.grad.detach().clone() for p in _params(a)]
    gen = torch.Generator().manual_seed(7)
    seeds = [_seed_state(name, _opt_of(b, p), p, gr, step0, gen) for p, gr in zip(_params(b), grads)]
    names = _kernel_names(lambda: b.train_dcll(x, y, regularize=False))
    for i, (p, (w0, m0, v0, st0), gr) in enumerate(zip(_params(b), seeds, grads)):
        opt = _opt_of(b, p)
        _check_rule("param %d" % i, name, opt, p.detach(), opt.state[p], w0, gr, m0, v0, st0)
    return a, b, names


# ------------------------------------------------------------------------------------------------------------------------
# 2: one step on every dispatch branch
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,hyper", CASES)
@pytest.mark.parametrize("case", sorted(OUT_CASES))
def test_output_layer_rule(case, name, hyper):
    c = OUT_CASES[case]
    _, b, names = _run(lambda: _conv(c), c.B, name, hyper)
    assert readout_branch(b.dclllayer, c.B, b.optimizer2) == c.branch
    _assert_opt_ran(names, c.branch, c.K)
    _assert_opt_ran(names, "wgrad+reduce_adam")


@pytest.mark.gpu
@pytest.mark.parametrize("name,hyper", CASES)
@pytest.mark.parametrize("case", sorted(I2H_CASES))
def test_i2h_conv_rule(case, name, hyper):
    c = I2H_CASES[case]
    _, b, names = _run(lambda: _conv(c), c.B, name, hyper)
    assert i2h_branch(b.dclllayer) == c.branch
    _assert_opt_ran(names, c.branch)


@pytest.mark.gpu
@pytest.mark.parametrize("name,hyper", CASES)
@pytest.mark.parametrize("B,n_in,n_out,K", DENSE_CASES)
def test_dense_rule(B, n_in, n_out, K, name, hyper):
    _, b, names = _run(lambda: _dense(n_in, n_out, K), B, name, hyper)
    _assert_opt_ran(names, "adam_flat")


def _apply_update_opt(lay, name, opt_i2h, opt_out, grads, batch):
    """dcll_conv_apply_update_opt through the C ABI on hand-given gradients, with the state of the two torch optimizers."""
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import _fill_optim, _store_optim
    desc = _lib.ConvLayer()
    lay._fill_desc(desc, batch, _lib.X_DENSE, None)
    args = _lib.TrainArgs()
    args.grad_w, args.grad_b, args.grad_wout, args.grad_bout = (_lib.ptr(t) for t in grads)
    rules = (_lib.Optim * 2)()
    sw = _fill_optim(args.adam_i2h, rules[0], opt_i2h, lay.i2h.weight, lay.i2h.bias)
    so = _fill_optim(args.adam_out, rules[1], opt_out, lay.output_.weight, lay.output_.bias)
    assert rules[0].kind == rules[1].kind != _lib.OPT_ADAM
    names = _kernel_names(lambda: _lib.check(_lib.lib.dcll_conv_apply_update_opt(ctypes.byref(desc), ctypes.byref(args),
                                                                                  rules, _lib.current_stream())))
    _store_optim(sw, args.adam_i2h, rules[0])
    _store_optim(so, args.adam_out, rules[1])
    return names


@pytest.mark.gpu
@pytest.mark.parametrize("name,hyper", CASES)
def test_conv_apply_update_rule(name, hyper):
    """dcll_conv_apply_update_opt (the gloo data-parallel update): parameters and state against float64 and torch, and the
    next forward sees the new weights."""
    hp, step0 = HYPERS[hyper]
    c = Case(2, 8, 3, (12, 12), None, 10, 4, True, "fp32", None)
    lay = _conv(c)
    lay.init_hiddens(c.B)
    st, x, _ = _inputs(lay, c.B, seed=3)
    params = [lay.i2h.weight, lay.i2h.bias, lay.output_.weight, lay.output_.bias]
    opt_i2h, opt_out = RULES[name](params[:2], **hp), RULES[name](params[2:], **hp)
    g = torch.Generator().manual_seed(4)
    grads = [(torch.randn(p.shape, generator=g) * 1e-3).cuda() for p in params]
    seeds = [_seed_state(name, o, p, gr, step0, g) for o, p, gr in zip((opt_i2h, opt_i2h, opt_out, opt_out), params, grads)]
    names = _apply_update_opt(lay, name, opt_i2h, opt_out, grads, c.B)
    torch.cuda.synchronize()
    assert any("opt_flat_kernel" in n for n in names) and not any("adam_flat_kernel" in n for n in names)
    for i, (o, p, (w0, m0, v0, st0), gr) in enumerate(zip((opt_i2h, opt_i2h, opt_out, opt_out), params, seeds, grads)):
        _check_rule("param %d" % i, name, o, p.detach(), o.state[p], w0, gr, m0, v0, st0)
    _set_state(lay, st)
    got = lay.forward(x)
    fresh = _conv(c, seed=9)
    fresh.load_state_dict(lay.state_dict())
    fresh.init_hiddens(c.B)
    _set_state(fresh, st)
    for u, w in zip(got, fresh.forward(x)):
        assert torch.equal(u, w)


# ------------------------------------------------------------------------------------------------------------------------
# 3 + 4: window drivers against per-step learn(); the host's step / mu_product chain against torch
# ------------------------------------------------------------------------------------------------------------------------
def _use_rule(net, name):
    """Every slice of `net` trains with torch.optim.<name> built as DCLLBase builds it (train.py's kwargs: betas (0, 0.95),
    weight decay 10, optimizer2 with lr 1e-4)."""
    for s in net.dcll_slices:
        lay = s.dclllayer
        s.optimizer = RULES[name](lay.i2h.parameters(), lr=float(s.optimizer.param_groups[0]["lr"]), betas=[0.0, 0.95],
                                  weight_decay=10)
        if lay.output_layer:
            s.optimizer2 = RULES[name](lay.output_.parameters(), lr=1e-4)


def _window_pair(name, precision):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_losses import _window_pair as wp
    (a, b), cells, tgt, y, T, burnin = wp(nn.SmoothL1Loss, precision)
    for n in (a, b):
        _use_rule(n, name)
        n.reset()
    return a, b, cells, tgt, y, T, burnin


def _assert_same_training(a, b, steps, name):
    for sa, sb in zip(a.dcll_slices, b.dcll_slices):
        la, lb = sa.dclllayer, sb.dclllayer
        assert torch.equal(la.i2h.weight, lb.i2h.weight) and torch.equal(la.i2h.bias, lb.i2h.bias)
        assert torch.equal(la.i2h.state.eps1, lb.i2h.state.eps1) and torch.equal(la.i2h.state.eps0, lb.i2h.state.eps0)
        assert np.array_equal(np.array(sa.clout), np.array(sb.clout)) and sa.iter == sb.iter
        pairs = [(sa.optimizer, sb.optimizer, la.i2h.weight, lb.i2h.weight), (sa.optimizer, sb.optimizer, la.i2h.bias, lb.i2h.bias)]
        if la.output_layer:
            assert torch.equal(la.output_.weight, lb.output_.weight) and torch.equal(la.output_.bias, lb.output_.bias)
            pairs.append((sa.optimizer2, sb.optimizer2, la.output_.weight, lb.output_.weight))
            pairs.append((sa.optimizer2, sb.optimizer2, la.output_.bias, lb.output_.bias))
        for oa, ob, pa, pb in pairs:
            wa, wb = oa.state[pa], ob.state[pb]
            assert sorted(wa) == sorted(wb)
            for k in wa:
                assert torch.equal(wa[k], wb[k]), k
            assert float(wb["step"]) == steps
            # 3: the chain depends on the step count only -- a torch optimizer stepped `steps` times on a CPU dummy
            p = nn.Parameter(torch.zeros(1))
            ref = type(ob)([p], **_kwargs(ob))
            for _ in range(steps):
                p.grad = torch.zeros(1)
                ref.step()
            assert torch.equal(wb["step"], ref.state[p]["step"])
            if name == "NAdam":
                assert torch.equal(wb["mu_product"], ref.state[p]["mu_product"])
        assert torch.isfinite(lb.i2h.weight).all()


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("precision", ["fp32", "f16x2"])
@pytest.mark.parametrize("name", sorted(RULES))
def test_window_equals_per_step(name, precision):
    a, b, cells, tgt, y, T, burnin = _window_pair(name, precision)
    for t in range(T):
        a.learn(cells[t], tgt[t])
    b.learn_window(cells, y)
    _assert_same_training(a, b, T - burnin + 1, name)


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(port, backend, out_q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    else:
        dist.init_process_group("gloo", rank=0, world_size=1)
    res = {}
    for name in sorted(RULES):
        try:
            a, b, cells, _, y, T, burnin = _window_pair(name, "f16x2")
            a.learn_window(cells, y)
            b.learn_window_dp(cells, y)
            torch.cuda.synchronize()
            _assert_same_training(a, b, T - burnin + 1, name)
            res[name] = "ok"
        except Exception as e:                      # reported by the parent test
            res[name] = repr(e)
    out_q.put(res)
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_data_parallel_single_rank_equals_learn_window(backend):
    """5: one rank of learn_window_dp (the C driver over NCCL, the per-layer Python loop over gloo) equals learn_window."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_dp_worker, args=(_free_port(), backend, q))
    p.start()
    res = q.get(timeout=900)
    p.join(timeout=120)
    assert res == {n: "ok" for n in RULES}, res


# ------------------------------------------------------------------------------------------------------------------------
# 6: the kernel-side weight images follow an _opt update
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RULES))
@pytest.mark.parametrize("case", ["bf16x3_rowpair", "bf16x3_layer0", "f16x2_rowpair"])
def test_next_forward_sees_updated_weights(case, name):
    c, lr = IMAGE_CASES[case]
    b = _slice(_conv(c), c.B, RULES[name], {"lr": lr, "weight_decay": 0.0})
    st, x, y = _inputs(b.dclllayer, c.B, seed=1)
    st2, x2, _ = _inputs(b.dclllayer, c.B, seed=2)
    before = [p.detach().clone() for p in _params(b)]
    _set_state(b.dclllayer, st)
    names = _kernel_names(lambda: b.train_dcll(x, y, regularize=False))
    _assert_opt_ran(names, i2h_branch(b.dclllayer))
    assert any(not torch.equal(p, q) for p, q in zip(_params(b), before))
    got = _next_forward(b, st2, x2)
    fresh = _slice(_conv(c, seed=9), c.B, None, {})
    fresh.load_state_dict(b.state_dict())
    want = _next_forward(fresh, st2, x2)
    for what, u, w in zip(("pvmem", "pvoutput", "spikes"), got, want):
        assert torch.equal(u, w), (what, float((u - w).abs().max()))


# ------------------------------------------------------------------------------------------------------------------------
# 7: optimizer.state_dict() after a device window drives a torch optimizer
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("name", sorted(RULES))
def test_state_dict_interchanges_with_torch(name):
    _, b, cells, _, y, T, burnin = _window_pair(name, "fp32")
    b.learn_window(cells, y)
    s = b.dcll_slices[-1]
    lay = s.dclllayer
    params = [lay.i2h.weight, lay.i2h.bias, lay.output_.weight, lay.output_.bias]
    opts = (s.optimizer, s.optimizer, s.optimizer2, s.optimizer2)
    # CPU copies of every parameter of the two optimizers, in their order (state_dict refers to parameters by position)
    cpu_of = {id(q): nn.Parameter(q.detach().cpu().clone()) for o in opts[1:3] for q in o.param_groups[0]["params"]}
    cpu = [cpu_of[id(p)] for p in params]
    torch_opts = tuple(RULES[name]([cpu_of[id(q)] for q in o.param_groups[0]["params"]], foreach=False) for o in opts[1:3])
    torch_opts[0].load_state_dict(s.optimizer.state_dict())
    torch_opts[1].load_state_dict(s.optimizer2.state_dict())
    g = torch.Generator().manual_seed(4)
    grads = [(torch.randn(p.shape, generator=g) * 1e-3).cuda() for p in params]
    before = [(p.detach().clone(), {k: v.clone() for k, v in o.state[p].items()}) for o, p in zip(opts, params)]
    _apply_update_opt(lay, name, s.optimizer, s.optimizer2, grads, lay.i2h.state.eps0.shape[0])
    for p, gr in zip(cpu, grads):
        p.grad = gr.cpu()
    for o in torch_opts:
        o.step()
    torch.cuda.synchronize()
    for i, (o, p, (w0, st0), gr, tp) in enumerate(zip(opts, params, before, grads, cpu)):
        assert float(o.state[p]["step"]) == T - burnin + 2
        tst = torch_opts[i // 2].state[tp]
        for k in st0:
            if k == "step" or k == "mu_product":
                assert torch.equal(o.state[p][k], tst[k]), (i, k)
            else:
                d = _ulp_dist(o.state[p][k], tst[k])
                assert int(d.max()) <= 1, (i, k, int(d.max()))
        mp = float(st0["mu_product"]) if name == "NAdam" else 1.0
        terms = _rule64(name, _group(o), w0, gr, st0["exp_avg"], st0[_vkey(name)], float(st0["step"]) + 1, mp)[5]
        tw = tp.detach().to(p.device).double()
        err, tol = (p.detach().double() - tw).abs(), 8 * EPS32 * terms + 2 * _ulp32(tw)
        assert not bool((err > tol).any()), (i, float((err / tol).max()))


# ------------------------------------------------------------------------------------------------------------------------
# 8 + 9: the training CLI; what stays unsupported fails loudly
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("optim_type", sorted(RULES))
def test_train_entry_point_with_optim_type(tmp_path, optim_type):
    from snn_modulation_classification_b200 import train
    args = ['--I_resolution', '16', '--Q_resolution', '16', '--burnin', '4', '--batch_size', '8', '--batch_size_test', '8',
            '--n_test_samples', '8', '--n_iters', '12', '--n_iters_test', '12', '--arp', '1.0', '--radio_ml_data_dir',
            str(tmp_path / 'no_such_dir'), '--synthetic', '--output', str(tmp_path / 'results'), '--n_steps', '2',
            '--n_test_interval', '1', '--optim_type', optim_type]
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        r = train.main(args)
    finally:
        os.chdir(cwd)
    assert type(r['net'].dcll_slices[0].optimizer).__name__ == optim_type
    p0, p1 = (torch.load(os.path.join(r['out_dir'], 'parameters_%d.pth' % i)) for i in (0, 1))
    for k in ('dcll_slices.0.dclllayer.i2h.weight', 'dcll_slices.2.dclllayer.i2h.weight', 'dcll_slices.2.dclllayer.output_.weight'):
        assert torch.isfinite(p1[k]).all() and not torch.equal(p0[k], p1[k]), k


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("make", [lambda ps: torch.optim.AdamW(ps, amsgrad=True), lambda ps: torch.optim.SGD(ps, lr=1e-3)],
                         ids=["AdamW_amsgrad", "SGD"])
def test_unsupported_optimizer_still_fails_loudly_in_the_windows(make):
    a, _, cells, _, y, _, _ = _window_pair("AdamW", "fp32")
    for s in a.dcll_slices:
        s.optimizer = make(list(s.dclllayer.i2h.parameters()))
    with pytest.raises(NotImplementedError, match="AdamW, Adamax, NAdam, RAdam"):
        a.learn_window(cells, y)
    with pytest.raises(NotImplementedError, match="AdamW, Adamax, NAdam, RAdam"):
        a.learn_window_dp(cells, y)
