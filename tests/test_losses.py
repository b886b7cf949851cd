"""Local losses computed on the device: every torch.nn class `train.py --loss_type` accepts with default arguments and
[B,K] one-hot float targets (DCLL_LOSS_*).  CPU: which criterion maps to which kind.  GPU (pytest -m gpu): gradients and
values against torch autograd, the window drivers against the per-step API bit for bit, the f16x2 gradient image with
cross-entropy, one rank of the data-parallel driver, and the training entry point."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 24

# the eight classes added to the three of the first release, and the element-wise / row-wise kinds they take
NEW_CLASSES = [nn.HuberLoss, nn.CrossEntropyLoss, nn.BCEWithLogitsLoss, nn.MultiLabelSoftMarginLoss, nn.SoftMarginLoss,
               nn.KLDivLoss, nn.PoissonNLLLoss, nn.HingeEmbeddingLoss]
NEW_KIND_CLASSES = [nn.CrossEntropyLoss, nn.BCEWithLogitsLoss, nn.SoftMarginLoss, nn.KLDivLoss, nn.PoissonNLLLoss,
                    nn.HingeEmbeddingLoss]
_ids = lambda classes: [c.__name__ for c in classes]


def _kinds():
    from snn_modulation_classification_b200 import _lib
    return {nn.SmoothL1Loss: _lib.LOSS_SMOOTHL1, nn.HuberLoss: _lib.LOSS_SMOOTHL1, nn.MSELoss: _lib.LOSS_MSE,
            nn.L1Loss: _lib.LOSS_L1, nn.CrossEntropyLoss: _lib.LOSS_CROSS_ENTROPY,
            nn.BCEWithLogitsLoss: _lib.LOSS_BCE_LOGITS, nn.MultiLabelSoftMarginLoss: _lib.LOSS_BCE_LOGITS,
            nn.SoftMarginLoss: _lib.LOSS_SOFT_MARGIN, nn.KLDivLoss: _lib.LOSS_KL_DIV,
            nn.PoissonNLLLoss: _lib.LOSS_POISSON_NLL, nn.HingeEmbeddingLoss: _lib.LOSS_HINGE}


def test_default_instances_map_to_device_kinds():
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import NATIVE_LOSSES, _loss_kind
    kinds = _kinds()
    assert sorted(NATIVE_LOSSES) == sorted(c.__name__ for c in kinds)
    for cls, kind in kinds.items():
        assert _loss_kind(cls()) == kind, cls.__name__
    assert (_lib.LOSS_SMOOTHL1, _lib.LOSS_MSE, _lib.LOSS_L1, _lib.LOSS_EXTERNAL) == (0, 1, 2, 3)
    assert _lib.ABI_VERSION == 12 and _lib.lib.dcll_abi_version() == 12


class _SubCE(nn.CrossEntropyLoss):
    pass


class _SubBCE(nn.BCEWithLogitsLoss):
    pass


@pytest.mark.parametrize("make", [
    lambda: nn.SmoothL1Loss(beta=0.5), lambda: nn.HuberLoss(delta=2.0), lambda: nn.MSELoss(reduction='sum'),
    lambda: nn.CrossEntropyLoss(label_smoothing=0.1), lambda: nn.CrossEntropyLoss(weight=torch.ones(K)),
    lambda: nn.CrossEntropyLoss(reduction='sum'), lambda: nn.BCEWithLogitsLoss(pos_weight=torch.ones(K)),
    lambda: nn.BCEWithLogitsLoss(weight=torch.ones(K)), lambda: nn.MultiLabelSoftMarginLoss(weight=torch.ones(K)),
    lambda: nn.SoftMarginLoss(reduction='none'), lambda: nn.KLDivLoss(log_target=True),
    lambda: nn.KLDivLoss(reduction='batchmean'), lambda: nn.PoissonNLLLoss(log_input=False),
    lambda: nn.PoissonNLLLoss(full=True), lambda: nn.HingeEmbeddingLoss(margin=2.0), _SubCE, _SubBCE, nn.NLLLoss,
    nn.BCELoss])
def test_other_arguments_and_subclasses_stay_external(make):
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import _loss_kind
    assert _loss_kind(make()) == _lib.LOSS_EXTERNAL


def test_per_step_kind_needs_a_target_shaped_like_the_readout():
    """Class-index targets for CrossEntropyLoss take the autograd route; the first three kinds keep their behaviour."""
    from snn_modulation_classification_b200 import _lib
    from snn_modulation_classification_b200.dcll.pytorch_libdcll import _step_loss_kind
    pred = torch.zeros(8, K)
    assert _step_loss_kind(nn.CrossEntropyLoss(), torch.zeros(8, K), pred) == _lib.LOSS_CROSS_ENTROPY
    assert _step_loss_kind(nn.CrossEntropyLoss(), torch.zeros(8, dtype=torch.long), pred) == _lib.LOSS_EXTERNAL
    assert _step_loss_kind(nn.SmoothL1Loss(), torch.zeros(1, K), pred) == _lib.LOSS_SMOOTHL1


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _rows(cls, B, seed):
    """Read-out rows x and targets y [B,K]: |x| ~ 100 in row 0 (|x| <= 8 for PoissonNLLLoss, whose value is exp(x)), the
    kinks d = x - y = +-1 in row 1, x = 1 exactly in row 2 (the hinge's kink for y = 0), ordinary values elsewhere;
    one-hot targets except the last row, a soft target summing to 0.7."""
    g = torch.Generator().manual_seed(seed)
    y = torch.zeros(B, K)
    y[torch.arange(B), torch.randint(0, K, (B,), generator=g)] = 1.0
    soft = torch.rand(K, generator=g)
    y[B - 1] = soft * (0.7 / float(soft.sum()))
    x = torch.randn(B, K, generator=g) * 1.5
    x[0] = (torch.rand(K, generator=g) * 2 - 1) * (8.0 if cls is nn.PoissonNLLLoss else 100.0)
    x[1] = y[1] + torch.where(torch.arange(K) % 2 == 0, 1.0, -1.0)
    x[2] = 1.0
    if cls is nn.KLDivLoss:
        x = -x.abs()        # log-probabilities: no cancellation in the value's sum
    return x, y


def _backward_both_routes(s, cls, y):
    """The native backward, then the autograd route (a subclass of the same class) from the same forward state: gradients
    left in .grad, no optimizer step.  Returns ((loss, grads) native, (loss, grads) autograd)."""
    lay = s.dclllayer
    params = [lay.i2h.weight, lay.i2h.bias] + ([lay.output_.weight, lay.output_.bias] if lay.output_layer else [])
    sub = type('Sub' + cls.__name__, (cls,), {})
    out = []
    for make in (cls, sub):
        s.crit, s.output_crit = make().cuda(), make().cuda()
        for p in params:
            p.grad = None
        loss = s._bwd_update(y, do_train=False)
        torch.cuda.synchronize()
        out.append((float(loss.reshape(-1)[0]), [p.grad.detach().clone() for p in params]))
    return out


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("cls", NEW_CLASSES, ids=_ids(NEW_CLASSES))
def test_conv_gradient_and_value_match_autograd(cls):
    from util_build import build_pair, rel_err
    B = 8
    net, _ = build_pair("radio_ml_conv", (1, 16, 16), B, K, arp=1.0, burnin=0)
    net.set_precision("fp32")
    net.reset()
    g = torch.Generator().manual_seed(3)
    inp = ((torch.rand(B, 1, 16, 16, generator=g) < 0.3).float()).cuda()
    for t in range(2):      # the second step sees traces and spikes in every layer
        inp_t = inp
        for i, s in enumerate(net.dcll_slices):
            out, _, _, _ = s.forward(inp_t, ignore_burnin=True)
            if t == 1:
                x, y = _rows(cls, B, seed=10 + i)
                outs = s.dclllayer._ctx[1]
                outs['pvoutput'].copy_(x.cuda())
                ref = cls()(x.cuda(), y.cuda())
                if s.dclllayer.output_layer:
                    x2, _ = _rows(cls, B, seed=20 + i)
                    outs['output'].copy_(x2.cuda())
                    ref = ref + cls()(x2.cuda(), y.cuda())
                (loss_n, g_n), (loss_a, g_a) = _backward_both_routes(s, cls, y.cuda())
                for j, (a, b) in enumerate(zip(g_n, g_a)):
                    assert rel_err(a, b) <= 2e-5, (i, j, rel_err(a, b))
                ref = float(ref)
                assert np.isfinite(loss_n) and abs(loss_n - ref) <= 1e-6 * abs(ref), (i, loss_n, ref, loss_a)
            inp_t = out


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("cls", NEW_CLASSES, ids=_ids(NEW_CLASSES))
def test_dense_gradient_matches_autograd(cls):
    from util_build import rel_err
    from snn_modulation_classification_b200.dcll import pytorch_libdcll as L
    B, In, Out = 8, 40, 32
    torch.manual_seed(0)
    lay = L.DenseDCLLlayer(In, Out, target_size=K).to("cuda").init_hiddens(B)
    s = L.DCLLClassification(dclllayer=lay, batch_size=B, loss=cls, optimizer=torch.optim.Adam,
                             kwargs_optimizer={"lr": 1e-6}, burnin=0)
    g = torch.Generator().manual_seed(1)
    for _ in range(2):
        s.forward((torch.rand(B, In, generator=g) < 0.3).float().cuda(), ignore_burnin=True)
    x, y = _rows(cls, B, seed=5)
    lay._ctx[1]['pvoutput'].copy_(x.cuda())
    (loss_n, g_n), (_, g_a) = _backward_both_routes(s, cls, y.cuda())
    for j, (a, b) in enumerate(zip(g_n, g_a)):
        assert float(b.abs().max()) > 0 and rel_err(a, b) <= 2e-5, (j, rel_err(a, b))
    assert abs(loss_n - float(cls()(x, y))) <= 1e-6 * abs(float(cls()(x, y)))


def _window_pair(cls, precision):
    from oracle import dcll_oracle as O
    from util_build import build_pair
    from snn_modulation_classification_b200.data.utils import iq2spiketrain
    B, T, W, burnin = 8, 12, 16, 4
    nets = []
    for _ in range(2):
        n, _ = build_pair("radio_ml_conv", (1, W, W), B, K, arp=1.0, burnin=burnin)
        n.set_precision(precision)
        for s in n.dcll_slices:
            s.crit, s.output_crit = cls().cuda(), cls().cuda()
        nets.append(n)
    g = torch.Generator().manual_seed(4)
    x = (torch.randn(B, 2, 1, 1024, generator=g) * 0.4).float()
    y = O.to_one_hot(torch.randint(0, K, (B,), generator=g), K).cuda()
    np.random.seed(1)
    cells, tgt = iq2spiketrain(x, y, out_w=W, out_h=W, max_duration=T, as_cells=True)
    return nets, cells, tgt, y, T, burnin


@pytest.mark.gpu
@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("precision", ["fp32", "f16x2"])
@pytest.mark.parametrize("cls", NEW_KIND_CLASSES, ids=_ids(NEW_KIND_CLASSES))
def test_window_equals_per_step(cls, precision):
    """learn_window computes the loss gradient in readout_finish_kernel, learn() in loss_grad_kernel: same bits."""
    (a, b), cells, tgt, y, T, burnin = _window_pair(cls, precision)
    a.reset()
    b.reset()
    for t in range(T):
        a.learn(cells[t], tgt[t])
    b.learn_window(cells, y)
    for sa, sb in zip(a.dcll_slices, b.dcll_slices):
        la, lb = sa.dclllayer, sb.dclllayer
        assert torch.equal(la.i2h.weight, lb.i2h.weight) and torch.equal(la.i2h.bias, lb.i2h.bias)
        assert torch.equal(la.i2h.state.eps1, lb.i2h.state.eps1) and torch.equal(la.i2h.state.arp, lb.i2h.state.arp)
        assert np.array_equal(np.array(sa.clout), np.array(sb.clout)) and len(sa.clout) == T - burnin + 1
        pairs = [(sa.optimizer, sb.optimizer, la.i2h.weight, lb.i2h.weight), (sa.optimizer, sb.optimizer, la.i2h.bias, lb.i2h.bias)]
        if la.output_layer:
            assert torch.equal(la.output_.weight, lb.output_.weight) and torch.equal(la.output_.bias, lb.output_.bias)
            pairs.append((sa.optimizer2, sb.optimizer2, la.output_.weight, lb.output_.weight))
        for oa, ob, pa, pb in pairs:
            wa, wb = oa.state[pa], ob.state[pb]
            assert float(wa["step"]) == float(wb["step"]) == T - burnin + 1
            assert torch.equal(wa["exp_avg"], wb["exp_avg"]) and torch.equal(wa["exp_avg_sq"], wb["exp_avg_sq"])
        assert torch.isfinite(la.i2h.weight).all()


@pytest.mark.gpu
@pytest.mark.parametrize("im,B", [((16, 16), 8), ((128, 128), 2)])
def test_f16x2_cross_entropy_gradient_image_does_not_saturate(im, B, monkeypatch):
    """Cross-entropy's sum_k |g_o| reaches 2/B, twice the bound the g_u image exponent assumes (inside its 2^4 slack): the
    f16x2 weight gradient must meet the bound tests/test_gpu_f16x2.py applies to SmoothL1 against the FP32 oracle."""
    from oracle import dcll_oracle as O
    from util_build import force_state, make_args, rel_err, state_dict_from_params
    from snn_modulation_classification_b200 import networks as N

    def ce_grad(pred, target, kind=None):
        p = pred.detach().clone().requires_grad_(True)
        nn.CrossEntropyLoss()(p, target).backward()
        return p.grad
    monkeypatch.setattr(O, "loss_grad", ce_grad)
    specs = O.make_specs(O.BUILTIN_SPECS["radio_ml_conv"], (1,) + im, K)
    params = O.random_params(specs, seed=2)
    sd = state_dict_from_params(params)
    net = N.ConvNetwork(make_args(0.0), (1,) + im, B, N.load_network_spec("radio_ml_conv"), K, act=torch.nn.Sigmoid(),
                        loss=torch.nn.CrossEntropyLoss, opt=torch.optim.SGD, opt_param={}, learning_rates=[0.0], burnin=0)
    net.load_state_dict(sd)
    net = net.to("cuda")
    net.reset(True)
    net.load_state_dict(sd)
    net.set_precision("f16x2")
    onet = O.OracleNet(specs, params, B, burnin=0)
    g = torch.Generator().manual_seed(5)
    x = (torch.rand(2, B, 1, *im, generator=g) < 0.1).float()
    y = O.to_one_hot(torch.randint(0, K, (B,), generator=g), K)
    for t in range(2):
        force_state(net, onet)
        fos, grads, inp = [], [], x[t]
        for i, sp in enumerate(specs):
            fo = O.conv_step_fwd(sp, params[i], onet.states[i], inp)
            grads.append(O.conv_local_grads(sp, params[i], fo, y))
            fos.append(fo)
            onet.states[i], inp = fo.state, fo.spikes
        for i, s in enumerate(net.dcll_slices):
            s.train_dcll(x[t].cuda() if i == 0 else fos[i - 1].spikes.cuda(), y.cuda(), regularize=False)
            assert rel_err(s.dclllayer.i2h.weight.grad, grads[i].gW) <= 1e-3, (t, i)
            assert rel_err(s.dclllayer.i2h.bias.grad, grads[i].gb) <= 5e-5, (t, i)
            if s.dclllayer.output_layer:
                assert rel_err(s.dclllayer.output_.weight.grad, grads[i].gWout) <= 5e-5, (t, i)


def _free_port():
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
    (a, b), cells, _, y, T, burnin = _window_pair(nn.CrossEntropyLoss, "f16x2")
    a.reset()
    b.reset()
    a.learn_window(cells, y)
    b.learn_window_dp(cells, y)
    torch.cuda.synchronize()
    ok = True
    for sa, sb in zip(a.dcll_slices, b.dcll_slices):
        la, lb = sa.dclllayer, sb.dclllayer
        ok = ok and torch.equal(la.i2h.weight, lb.i2h.weight) and torch.equal(la.i2h.bias, lb.i2h.bias)
        ok = ok and torch.equal(la.i2h.state.eps1, lb.i2h.state.eps1)
        ok = ok and np.array_equal(np.array(sa.clout), np.array(sb.clout)) and sa.iter == sb.iter
        if la.output_layer:
            ok = ok and torch.equal(la.output_.weight, lb.output_.weight) and torch.equal(la.output_.bias, lb.output_.bias)
        wa, wb = sa.optimizer.state[la.i2h.weight], sb.optimizer.state[lb.i2h.weight]
        ok = ok and float(wa["step"]) == float(wb["step"]) == T - burnin + 1 and torch.equal(wa["exp_avg_sq"], wb["exp_avg_sq"])
    out_q.put(ok)
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_data_parallel_single_rank_cross_entropy_equals_learn_window(backend):
    """One rank of learn_window_dp (the C driver over NCCL, the per-layer Python loop over gloo) with CrossEntropyLoss
    reproduces learn_window bit for bit: the all-reduce of one rank is the identity."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_dp_worker, args=(_free_port(), backend, q))
    p.start()
    ok = q.get(timeout=600)
    p.join(timeout=120)
    assert ok


@pytest.mark.gpu
@pytest.mark.parametrize("loss_type", ["CrossEntropyLoss", "BCEWithLogitsLoss"])
def test_train_entry_point_with_loss_type(tmp_path, loss_type):
    from snn_modulation_classification_b200 import train
    args = ['--I_resolution', '16', '--Q_resolution', '16', '--burnin', '4', '--batch_size', '8', '--batch_size_test', '8',
            '--n_test_samples', '8', '--n_iters', '12', '--n_iters_test', '12', '--arp', '1.0', '--radio_ml_data_dir',
            str(tmp_path / 'no_such_dir'), '--synthetic', '--output', str(tmp_path / 'results'), '--n_steps', '2',
            '--n_test_interval', '1', '--loss_type', loss_type]
    os.chdir(tmp_path)
    r = train.main(args)
    assert type(r['net'].dcll_slices[0].crit).__name__ == loss_type
    p0, p1 = (torch.load(os.path.join(r['out_dir'], 'parameters_%d.pth' % i)) for i in (0, 1))
    for k in ('dcll_slices.0.dclllayer.i2h.weight', 'dcll_slices.2.dclllayer.i2h.weight', 'dcll_slices.2.dclllayer.output_.weight'):
        assert torch.isfinite(p1[k]).all() and not torch.equal(p0[k], p1[k]), k
    assert np.isfinite(r['acc_test']).all()


@pytest.mark.gpu
def test_unsupported_variant_still_fails_loudly_in_the_windows():
    (a, _), cells, _, y, _, _ = _window_pair(nn.CrossEntropyLoss, "fp32")
    for s in a.dcll_slices:
        s.crit, s.output_crit = nn.CrossEntropyLoss(label_smoothing=0.1), nn.CrossEntropyLoss(label_smoothing=0.1)
    a.reset()
    with pytest.raises(NotImplementedError, match="CrossEntropyLoss"):
        a.learn_window(cells, y)
    with pytest.raises(NotImplementedError, match="CrossEntropyLoss"):
        a.learn_window_dp(cells, y)
