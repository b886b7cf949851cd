"""Pins the oracle against the LIVE reference (the checkout of the original project named by DCLL_REFERENCE_ROOT or
BASELINE.json's reference_path, or its vendored copy oracle/_ref; skipped without one).

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so
"the reference classes executed on the same inputs and seeds" is the definition
of parity.  tests/golden/ holds the same comparisons frozen as fixtures so they
also run where the reference is absent.
"""
import copy

import numpy as np
import pytest
import torch

from oracle import dcll_oracle as O
from oracle import refshim

pytestmark = [pytest.mark.reference,
              pytest.mark.skipif(not refshim.reference_available(), reason="reference not present")]


def synth_iq(B, N=1024, seed=1):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 2, 1, N, generator=g) * 0.4).float()


@pytest.mark.parametrize("W,B,T", [(16, 64, 96), (128, 64, 64), (28, 32, 40)])
@pytest.mark.parametrize("gamma", [True, False])
def test_encoder_cells_match_reference(W, B, T, gamma):
    _, _, U = refshim.load_reference()
    x = synth_iq(B)
    y = O.to_one_hot(torch.arange(B) % 24, 24)
    np.random.seed(3)
    frames, tgt = U.iq2spiketrain(x, y, out_w=W, out_h=W, max_duration=T, do_gamma=gamma)
    np.random.seed(3)
    t_start = np.random.randint(0, 1024 - T + 1)
    cells = O.encode_cells(x.numpy(), W, W, t_start=t_start, max_duration=T, do_gamma=gamma)
    assert frames.sum() == T * B                      # exactly one spike per (t, b)
    mine = O.cells_to_frames(cells, W, W, dtype=np.float64)
    assert np.array_equal(mine, frames)
    assert np.array_equal(O.repeat_targets(y, T), tgt)


def test_encoder_nondefault_bounds():
    _, _, U = refshim.load_reference()
    x = synth_iq(32, seed=7) * 2
    y = O.to_one_hot(torch.zeros(32, dtype=torch.int64), 24)
    np.random.seed(0)
    frames, _ = U.iq2spiketrain(x, y, out_w=20, out_h=12, min_I=-1.5, max_I=0.7, min_Q=-0.3, max_Q=2.0,
                                max_duration=1024)
    cells = O.encode_cells(x.numpy(), 20, 12, -1.5, 0.7, -0.3, 2.0, 0, 1024)
    assert np.array_equal(O.cells_to_frames(cells, 12, 20, np.float64), frames)


CASES = [
    # spec, im_dims, B, K, arp, burnin, steps
    ("radio_ml_conv", (1, 16, 16), 8, 24, 0.0, 3, 8),
    ("radio_ml_conv", (1, 16, 16), 8, 24, 1.0, 3, 8),
    ("mnist_conv", (1, 28, 28), 6, 10, 0.0, 2, 6),
    ("radio_ml_conv_ref", (1, 4, 128), 2, 24, 0.0, 2, 4),
]


def _inputs(im_dims, B, K, steps, seed=5):
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(steps, B, *im_dims, generator=g) < 0.1).float()
    y = O.to_one_hot(torch.randint(0, K, (B,), generator=g), K)
    return x, y


def _close_in_steps(ref_p, mine, lr, max_frac=5e-2, mean_frac=2e-4):
    d = (ref_p.detach() - mine).abs()
    assert d.max() <= max_frac * lr, (float(d.max()) / lr)
    assert d.mean() <= mean_frac * lr, (float(d.mean()) / lr)


def _sync_from_reference(slice_, onet, i):
    lay, p, sl = slice_.dclllayer, onet.params[i], onet.slots[i]
    pairs = [(lay.i2h.weight, p.weight, "w", slice_.optimizer), (lay.i2h.bias, p.bias, "b", slice_.optimizer)]
    if lay.output_layer:
        pairs += [(lay.output_.weight, p.wout, "wout", slice_.optimizer2),
                  (lay.output_.bias, p.bout, "bout", slice_.optimizer2)]
    for ref_p, mine, key, opt in pairs:
        mine.copy_(ref_p.detach())
        stt = opt.state[ref_p]
        sl[key].exp_avg.copy_(stt["exp_avg"])
        sl[key].exp_avg_sq.copy_(stt["exp_avg_sq"])
        assert sl[key].step == int(stt["step"])


@pytest.mark.parametrize("backend", ["closed", "autograd"])
@pytest.mark.parametrize("spec,im_dims,B,K,arp,burnin,steps", CASES)
def test_training_matches_reference(spec, im_dims, B, K, arp, burnin, steps, backend):
    net = refshim.build_reference_net(spec, im_dims, B, K, arp=arp, burnin=burnin)
    specs = O.make_specs(O.BUILTIN_SPECS[spec], im_dims, K, wrp=arp)
    params = O.params_from_state_dict(copy.deepcopy(net.state_dict()), len(specs))
    onet = O.OracleNet(specs, params, B, burnin=burnin, backend=backend)
    x, y = _inputs(im_dims, B, K, steps)
    net.reset()
    net.train()
    onet.reset()
    lr = 1e-6
    for t in range(steps):
        net.learn(x[t], y)
        onet.learn(x[t], y)
        for i, s in enumerate(net.dcll_slices):
            st = s.dclllayer.i2h.state
            assert torch.equal(st.eps0, onet.states[i].eps0)
            assert torch.equal(st.eps1, onet.states[i].eps1)
            if arp > 0:
                assert torch.equal(st.arp, onet.states[i].arp)
            lay, p = s.dclllayer, onet.params[i]
            if backend == "autograd":
                assert torch.equal(lay.i2h.weight.detach(), p.weight.detach())
                assert torch.equal(lay.i2h.bias.detach(), p.bias.detach())
                if lay.output_layer:
                    assert torch.equal(lay.output_.weight.detach(), p.wout.detach())
                continue
            # closed form differs from autograd only by summation order in the conv weight
            # gradient; the Adam step is O(lr) whatever |g| is, so the tolerance is in units of lr.
            # Training is chaotic (error x2 per step, DESIGN.md), so the comparison is
            # teacher-forced: weights and Adam moments are re-synchronised after every step.
            # Elements whose gradient nearly cancels against weight_decay*w see the rounding of gW
            # amplified by 1/sqrt(v), hence a loose max bound next to a tight mean bound.
            _close_in_steps(lay.i2h.weight, p.weight, lr)
            _close_in_steps(lay.i2h.bias, p.bias, lr)
            if lay.output_layer:
                _close_in_steps(lay.output_.weight, p.wout, 1e-4)
                _close_in_steps(lay.output_.bias, p.bout, 1e-4)
            if t + 1 >= burnin:
                _sync_from_reference(s, onet, i)
    labels = torch.stack([y] * steps)
    assert net.accuracy(labels) == onet.accuracy(labels.numpy())
    for i, s in enumerate(net.dcll_slices):
        assert len(s.clout) == len(onet.clout[i]) == steps - burnin + 1
        assert np.array_equal(np.array(s.clout), np.array(onet.clout[i]))


@pytest.mark.parametrize("spec,im_dims,B,K,arp,burnin,steps", CASES[:3])
def test_closed_form_grads_match_autograd(spec, im_dims, B, K, arp, burnin, steps):
    """g_o/gW/gb/gWout of the closed form vs autograd on the reference layer (single step)."""
    net = refshim.build_reference_net(spec, im_dims, B, K, arp=arp, burnin=0)
    specs = O.make_specs(O.BUILTIN_SPECS[spec], im_dims, K, wrp=arp)
    params = O.params_from_state_dict(copy.deepcopy(net.state_dict()), len(specs))
    x, y = _inputs(im_dims, B, K, 3)
    spikes = x[0]
    for i, s in enumerate(net.dcll_slices):
        lay = s.dclllayer
        st = O.zero_state(specs[i], B)
        # two warm steps so traces are non-trivial
        for t in range(2):
            lay.forward(x[t] if i == 0 else spikes)
            fo = O.conv_step_fwd(specs[i], params[i], st, x[t] if i == 0 else spikes)
            st = fo.state
        lay.zero_grad()
        o, pvo, pv, pvmem = lay.forward(x[2] if i == 0 else spikes)
        loss = s.crit(pvo, y)
        if lay.output_layer:
            loss = loss + s.output_crit(o, y)
        loss.backward()
        fo = O.conv_step_fwd(specs[i], params[i], st, x[2] if i == 0 else spikes)
        g = O.conv_local_grads(specs[i], params[i], fo, y)
        assert torch.equal(fo.pvoutput, pvo.detach())
        assert torch.equal(fo.pvmem, pvmem.detach())
        torch.testing.assert_close(g.gW, lay.i2h.weight.grad, rtol=1e-4, atol=1e-6 * float(g.gW.abs().max()))
        torch.testing.assert_close(g.gb, lay.i2h.bias.grad, rtol=1e-4, atol=1e-6 * float(g.gb.abs().max()))
        if lay.output_layer:
            torch.testing.assert_close(g.gWout, lay.output_.weight.grad, rtol=1e-5, atol=1e-9)
            torch.testing.assert_close(g.gbout, lay.output_.bias.grad, rtol=1e-5, atol=1e-9)
        spikes = fo.spikes


def test_inference_matches_reference():
    B, K, T = 8, 24, 12
    net = refshim.build_reference_net("radio_ml_conv", (1, 16, 16), B, K, arp=1.0, train=False)
    specs = O.make_specs(O.BUILTIN_SPECS["radio_ml_conv"], (1, 16, 16), K, wrp=1.0)
    onet = O.OracleNet(specs, O.params_from_state_dict(net.state_dict(), 3), B)
    x, y = _inputs((1, 16, 16), B, K, T)
    net.reset()
    net.eval()
    onet.reset()
    for t in range(T):
        net.test(x[t])
        onet.test(x[t])
    for i, s in enumerate(net.dcll_slices):
        assert np.array_equal(np.array(s.clout), np.array(onet.clout[i]))
        assert torch.equal(s.dclllayer.i2h.state.eps1, onet.states[i].eps1)
    labels = torch.stack([y] * T)
    assert net.accuracy(labels) == onet.accuracy(labels.numpy())
    assert np.array_equal(net.confusion_matrix(labels), O.confusion_matrix(onet.clout[-1], labels.numpy(), K))


def test_dense_layer_matches_reference():
    L, _, _ = refshim.load_reference()
    torch.manual_seed(0)
    np.random.seed(0)
    for wrp in (0.0, 2.0):
        with refshim.quiet():
            lay = L.DenseDCLLlayer(40, 24, target_size=10, wrp=wrp, random_tau=True).init_hiddens(5)
        m = lay.i2h
        p = O.ConvParams(m.weight.detach().clone(), m.bias.detach().clone(), m.alpha.clone(), m.alphas.clone(),
                         m.tau_m__dt.clone(), m.tau_s__dt.clone(), lay.i2o.weight.clone(), lay.i2o.bias.clone())
        st = O.ConvState(torch.zeros(5, 40), torch.zeros(5, 40), torch.zeros(5, 24) if wrp > 0 else None)
        y = O.to_one_hot(torch.arange(5), 10)
        for t in range(4):
            x = (torch.rand(5, 40) < 0.3).float()
            lay.zero_grad()
            o, pvo, pv, vm = lay.forward(x)
            torch.nn.SmoothL1Loss()(pvo, y).backward()
            fo = O.dense_step_fwd(p, st, x, wrp=wrp)
            st = fo.state
            assert torch.equal(fo.vmem, vm.detach()) and torch.equal(fo.spikes, o)
            assert torch.equal(fo.pvoutput, pvo.detach())
            _, _, gW, gb = O.dense_local_grads(p, fo, y)
            torch.testing.assert_close(gW, m.weight.grad, rtol=1e-4, atol=1e-7 * float(gW.abs().max()))
            torch.testing.assert_close(gb, m.bias.grad, rtol=1e-4, atol=1e-7 * float(gb.abs().max()))


def test_image2spiketrain_matches_reference():
    """data/utils.py:15-40 -- same numpy stream, same spikes (incl. a non-default min_duration: ragged T_i)."""
    _, _, U = refshim.load_reference()
    g = torch.Generator().manual_seed(3)
    x = torch.rand(6, 1, 7, 5, generator=g)
    y = O.to_one_hot(torch.randint(0, 10, (6,), generator=g), 10).numpy()
    for kw in (dict(gain=100, max_duration=40), dict(gain=50, min_duration=10, max_duration=33)):
        np.random.seed(11)
        want, want_t = U.image2spiketrain(x, y, (1, 7, 5), **kw)
        np.random.seed(11)
        got, got_t = O.image2spiketrain(x, y, (1, 7, 5), **kw)
        assert got.shape == want.shape and np.array_equal(got, want) and np.array_equal(got_t, want_t)
        assert 0 < got.mean() < 0.2
