"""Network assembly: mirror of the reference's ``networks/__init__.py`` (ref lines cited inline).

``ConvNetwork`` keeps the reference API (``learn`` / ``test`` / ``reset`` / ``accuracy`` /
``confusion_matrix`` / ``write_stats``, ``dcll_slices`` ModuleList, state_dict keys) and adds
``learn_window`` / ``test_window``: the whole T-loop of train.py:249-251 / test_radio_ml.py:144-145 in one
C call (``dcll_net_window``), with no per-timestep Python, host sync or allocation.
"""
import ctypes
import os
from ast import literal_eval as make_tuple

import torch
import yaml

from .. import _lib
from ..dcll.pytorch_libdcll import (NATIVE_LOSSES, Conv2dDCLLlayer, DCLLClassification, SpikeCells, _as_cuda_f32,
                                    _fill_adam, _is_plain_adam, _loss_kind, _store_steps, device,
                                    DEVICE_OPTIMIZERS, _fill_optim, _on_device, _optims_of, _store_optim)

_HERE = os.path.dirname(os.path.abspath(__file__))

# Values of the reference's networks/*.yaml, available by name so that nothing needs the reference tree.
BUILTIN_SPECS = {
    'radio_ml_conv': [dict(out_channels=32, kernel_size=7, padding=3, pooling=1) for _ in range(3)],
    'mnist_conv': [dict(out_channels=16, kernel_size=7, padding=2, pooling=2),
                   dict(out_channels=24, kernel_size=7, padding=2, pooling=1),
                   dict(out_channels=32, kernel_size=7, padding=2, pooling=2)],
    'radio_ml_conv_ref': [dict(out_channels=64, kernel_size=(1, 3), padding=(0, 1), pooling=(1, 2))
                          for _ in range(7)],
}


def load_network_spec(yaml_path):
    """ref:10-18.  ``yaml_path``: a YAML file with the reference's schema
    (``conv_layers: [{out_channels, kernel_size, padding, pooling}]``, ints or tuple strings such as
    "(1, 3)"), or the bare name of a built-in spec ('radio_ml_conv', 'mnist_conv', 'radio_ml_conv_ref')."""
    key = os.path.splitext(os.path.basename(str(yaml_path)))[0]
    if not os.path.isfile(yaml_path):
        local = os.path.join(_HERE, key + '.yaml')
        if os.path.isfile(local):
            yaml_path = local
        elif key in BUILTIN_SPECS:
            return [dict(c) for c in BUILTIN_SPECS[key]]
        else:
            raise FileNotFoundError(yaml_path)
    with open(yaml_path, 'r') as f:
        network_spec = yaml.safe_load(f)
    convs = network_spec['conv_layers']
    for layer_spec in convs:
        for k, v in layer_spec.items():
            if type(v) != int:
                layer_spec[k] = make_tuple(v)      # e.g. the string "(2, 0)" -> (2, 0)
    return convs


_DP_HANDLES = {}
STACK16_F16X2_MAX_BATCH = 4096      # largest batch for which test_window runs dcll_infer_stack16 in 'f16x2'


def grad_bucket(lay, dev):
    """One flat float32 bucket per layer holding (gW, gb[, gWout, gbout]) back to back: the unit of the
    data-parallel all-reduce (SURVEY section 8e: 6.4 KB for conv0, 201 KB for conv1/2, + 24*F+24 floats for
    output_).  Returns (flat, views)."""
    sizes = [lay.i2h.weight.numel(), lay.i2h.bias.numel()]
    if lay.output_layer:
        sizes += [lay.output_.weight.numel(), lay.output_.bias.numel()]
    flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
    return flat, list(flat.split(sizes))


def allreduce_mean(flat, group=None, async_op=False):
    """Average a gradient bucket over the ranks.  Every rank normalises its local loss by its own B_local*K
    (mean reduction), shards are equal, so the mean of the per-rank gradients is the global-batch gradient.
    NCCL averages in the collective; other backends (gloo in the CPU tests) sum and divide."""
    import torch.distributed as dist
    if dist.get_backend(group) == 'nccl':
        return dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=False)   # completed when it returns
    flat.div_(dist.get_world_size(group))
    return None


class ConvNetwork(torch.nn.Module):
    def __init__(self, args, im_dims, batch_size, convs, target_size, act, loss, opt, opt_param, learning_rates,
                 DCLLSlice=DCLLClassification, burnin=50):
        super(ConvNetwork, self).__init__()
        self.batch_size = batch_size
        self.num_layers = len(convs)
        self.dcll_slices = torch.nn.ModuleList()
        n = im_dims
        for i, conf in enumerate(convs):                                # ref:148-172
            layer = Conv2dDCLLlayer(in_channels=n[0],
                                    out_channels=int(conf['out_channels'] * args.netscale),
                                    kernel_size=conf['kernel_size'], padding=conf['padding'],
                                    pooling=conf['pooling'], im_dims=n[1:3], target_size=target_size,
                                    alpha=args.alpha, alphas=args.alphas, alpharp=args.alpharp, wrp=args.arp,
                                    act=act, lc_ampl=args.lc_ampl, random_tau=args.random_tau, spiking=True,
                                    lc_dropout=False, output_layer=(i == self.num_layers - 1)
                                    ).to(device).init_hiddens(batch_size)
            n = torch.Size([layer.out_channels]) + layer.output_shape
            layer_opt_param = opt_param.copy()
            if learning_rates is not None:
                layer_opt_param['lr'] = learning_rates[min(i, len(learning_rates) - 1)]
            self.dcll_slices.append(DCLLSlice(dclllayer=layer, name='conv%d' % i, batch_size=batch_size, loss=loss,
                                              optimizer=opt, kwargs_optimizer=layer_opt_param, collect_stats=True,
                                              burnin=burnin))
        self._win = None
        # the training / inference CLIs' --precision (a mode of the layers, not a parameter: it survives .to() and
        # load_state_dict); callers whose args carry none keep 'fp32'
        self.set_precision(getattr(args, 'precision', 'fp32'))

    def set_precision(self, mode):
        """'fp32': FP32-exact parity mode (CUDA-core FMA).  'bf16x3': convolutions of the layers with an
        instantiated tensor-core shape run on tcgen05 with split-bf16 operands (3 MMAs, FP32 accumulation in TMEM);
        pooled layers fall back to FP32 per layer.  'f16x2': the same kernels with the trace operand (eps1, in [0,1]) as ONE fp16
        value against split-bf16 weights / local gradients -- two products instead of three and no lo pass over the traces
        (membrane error ~1e-4 of its scale instead of ~1e-5; spike-flip rate within the 1e-3 bound of the headline mode)."""
        if mode not in ('fp32', 'bf16x3', 'f16x2'):
            raise ValueError("precision must be 'fp32', 'bf16x3' or 'f16x2'")
        for s in self.dcll_slices:
            lay = s.dclllayer
            lay.i2h.precision = mode if max(lay.pooling) == 1 else 'fp32'
            lay.i2h._wt_key = None
        return self

    # -- reference per-timestep API -------------------------------------------------------------
    def learn(self, x, labels):                                         # ref:175-180
        spikes = x
        for s in self.dcll_slices:
            spikes, _, _, _, _ = s.train_dcll(spikes, labels, regularize=False)

    def test(self, x):                                                  # ref:182-185
        spikes = x
        for s in self.dcll_slices:
            spikes, _, _, _ = s.forward(spikes, ignore_burnin=True)

    def reset(self, init_states=False):                                 # ref:187-189
        for s in self.dcll_slices:
            s.init(self.batch_size, init_states=init_states)

    def write_stats(self, writer, epoch, comment=''):                   # ref:191-193
        for s in self.dcll_slices:
            s.write_stats(writer, label='test' + comment, epoch=epoch)

    def accuracy(self, labels):                                         # ref:195-196
        return [s.accuracy(labels) for s in self.dcll_slices]

    def confusion_matrix(self, labels):                                 # ref:198-199
        return self.dcll_slices[-1].confusion_matrix(labels)

    # -- whole-window fast path --------------------------------------------------------------------
    def _window_buffers(self, batch):
        key = (batch, self.dcll_slices[0].dclllayer.i2h.weight.device)
        if self._win is not None and self._win['key'] == key:
            return self._win
        dev = key[1]
        outs = []
        for s in self.dcll_slices:
            lay = s.dclllayer
            hp, wp = lay.get_output_shape()
            pooled = (batch, lay.out_channels, hp, wp)
            outs.append(dict(spikes=torch.empty(pooled, device=dev), pv=torch.empty(pooled, device=dev), pvmem=None,
                             pvoutput=torch.empty((batch, lay.target_size), device=dev),
                             output=torch.empty((batch, lay.target_size), device=dev) if lay.output_layer else None))
        self._win = dict(key=key, outs=outs)
        return self._win

    def _run_window(self, x, labels, train):
        """x: dense spikes [T,B,C,H,W] (tensor) or SpikeCells-like (cells [T,B,2]); labels [B,K] or [T,B,K]."""
        n = self.num_layers
        if isinstance(x, SpikeCells):
            x_t, x_mode = x.cells, _lib.X_CELLS
            T, batch = int(x_t.shape[0]), int(x_t.shape[1])
        else:
            x_t, x_mode = _as_cuda_f32(x), _lib.X_DENSE
            T, batch = int(x_t.shape[0]), int(x_t.shape[1])
        for s in self.dcll_slices:
            i2h = s.dclllayer.i2h
            if i2h.state.eps0.shape[0] != batch:
                import logging
                logging.warning("Batch size changed from {} to {} since last iteration. Reallocating states."
                                .format(i2h.state.eps0.shape[0], batch))
                i2h.init_state(batch, s.dclllayer.im_dims)
        win = self._window_buffers(batch)
        Layers, Trains = _lib.ConvLayer * n, _lib.TrainArgs * n
        layers, trains = Layers(), Trains()
        olds, states = [], []
        rules = self._window_rules('learn_window', 'use learn() per timestep') if train else None
        for i, s in enumerate(self.dcll_slices):
            old, _ = s.dclllayer._fill_desc(layers[i], batch, x_mode if i == 0 else _lib.X_DENSE, win['outs'][i])
            olds.append(old)
            if train:
                lay = s.dclllayer
                kind = _loss_kind(s.crit)
                if kind == _lib.LOSS_EXTERNAL:
                    raise NotImplementedError('learn_window implements %s with default arguments; use learn()'
                                              % ', '.join(NATIVE_LOSSES))
                trains[i].loss_kind, trains[i].apply_update = kind, 1
                states.append(self._fill_slice(i, trains[i], rules))
        target, t_stride = None, 0
        if labels is not None:
            target = _as_cuda_f32(labels)
            if target.dim() == 3:
                # [T,B,K] time-varying labels, or [1,B,K] = one row for the whole window; anything else would make the
                # driver read past the end of the buffer.  No device->host comparison here (no host sync in the window).
                if target.shape[0] == 1:
                    t_stride = 0
                elif target.shape[0] == T:
                    t_stride = target.shape[1] * target.shape[2]
                else:
                    raise ValueError('labels [T,B,K] must cover the window: got %d rows for T = %d'
                                     % (target.shape[0], T))
            if tuple(target.shape[-2:]) != (batch, int(self.dcll_slices[0].dclllayer.target_size)):
                raise ValueError('labels must be [B,K] or [T,B,K] with B = %d, K = %d; got %s'
                                 % (batch, int(self.dcll_slices[0].dclllayer.target_size), tuple(target.shape)))
        iter0 = (ctypes.c_int32 * n)(*[int(s.iter) for s in self.dcll_slices])
        clout = torch.empty((T, n, batch), dtype=torch.int32, device=x_t.device)
        burnin = int(self.dcll_slices[0].burnin)
        # activity statistics (DCLLBase.forward :658-661): 19-bin pv histogram every 20 iterations, kept on the device
        collect = any(getattr(s, 'collect_stats', False) for s in self.dcll_slices)
        hist_cap = T // 20 + 1
        hist = torch.zeros((n, hist_cap, 19), dtype=torch.int32, device=x_t.device) if collect else None
        if rules is not None:
            _lib.check(_lib.lib.dcll_net_window_stats_opt(layers, trains, rules, n, _lib.ptr(x_t), _lib.ptr(target), t_stride, T,
                                                          1, burnin, iter0, _lib.ptr(clout), _lib.ptr(hist),
                                                          20 if collect else 0, hist_cap, _lib.current_stream()))
        else:
            _lib.check(_lib.lib.dcll_net_window_stats(layers, trains if train else None, n, _lib.ptr(x_t), _lib.ptr(target),
                                                      t_stride, T, 1 if train else 0, burnin, iter0, _lib.ptr(clout),
                                                      _lib.ptr(hist), 20 if collect else 0, hist_cap, _lib.current_stream()))
        for i, s in enumerate(self.dcll_slices):
            s.dclllayer.i2h._commit_state(*olds[i], flips=T)
            s.dclllayer._ctx = None
            # DCLLClassification.forward counting rule (ref:724): rows with ignore_burnin or iter >= burnin
            first = 0 if not train else max(0, int(s.burnin) - int(s.iter) - 1)
            if first < T:
                s.clout.extend(clout[first:, i, :])
            if collect and s.collect_stats:
                n_h = (int(s.iter) + T) // 20 - int(s.iter) // 20        # iterations with iter % 20 == 0 in this window
                for j in range(n_h):
                    s.activity_hist.append(hist[i, j].float())
            s.iter += T
            if train:
                self._store_slice(i, trains[i], rules, states[i])
        return clout

    def _window_rules(self, who, hint=''):
        """None when every slice trains with plain Adam (the Adam entry points); else the dcll_optim array [2 n] of the _opt
        entry points, when every optimizer is one the device applies.  Raises NotImplementedError otherwise."""
        opts = [o for s in self.dcll_slices for o in _optims_of(s)]
        if all(_is_plain_adam(o) for o in opts):
            return None
        if not _on_device(*opts):
            raise NotImplementedError('%s needs %s slices (torch.optim classes, one param group, no amsgrad / maximize / '
                                      'capturable / differentiable, a float lr)%s'
                                      % (who, ', '.join(DEVICE_OPTIMIZERS), '; ' + hint if hint else ''))
        return (_lib.Optim * (2 * self.num_layers))()

    def _fill_slice(self, i, train, rules):
        """dcll_adam (+ dcll_optim) of slice i's optimizers; returns their states."""
        s = self.dcll_slices[i]
        lay = s.dclllayer
        if rules is None:
            st = [_fill_adam(train.adam_i2h, s.optimizer, lay.i2h.weight, lay.i2h.bias)]
            if lay.output_layer:
                st.append(_fill_adam(train.adam_out, s.optimizer2, lay.output_.weight, lay.output_.bias))
            return st
        st = [_fill_optim(train.adam_i2h, rules[2 * i], s.optimizer, lay.i2h.weight, lay.i2h.bias)]
        if lay.output_layer:
            st.append(_fill_optim(train.adam_out, rules[2 * i + 1], s.optimizer2, lay.output_.weight, lay.output_.bias))
        return st

    def _store_slice(self, i, train, rules, states):
        if rules is None:
            _store_steps(states[0], train.adam_i2h.step)
            if self.dcll_slices[i].dclllayer.output_layer:
                _store_steps(states[1], train.adam_out.step)
            return
        _store_optim(states[0], train.adam_i2h, rules[2 * i])
        if self.dcll_slices[i].dclllayer.output_layer:
            _store_optim(states[1], train.adam_out, rules[2 * i + 1])

    def _dp_handle(self, group, max_ctas):
        """The raw-NCCL communicator of the C driver for `group` (created once: rank 0 draws the unique id, the ranks receive
        it through torch.distributed, every rank joins)."""
        import torch.distributed as dist
        key = (id(group), dist.get_rank(group), dist.get_world_size(group), int(max_ctas))
        if key in _DP_HANDLES:                     # one communicator per (group, CTA cap) and process, shared by all networks
            return _DP_HANDLES[key]
        lib_path = _lib.nccl_library_path()
        lib_c = lib_path.encode() if lib_path else None
        dev = self.dcll_slices[0].dclllayer.i2h.weight.device
        uid = torch.zeros(128, dtype=torch.uint8)
        if dist.get_rank(group) == 0:
            buf = (ctypes.c_uint8 * 128)()
            _lib.check(_lib.lib.dcll_dp_unique_id(lib_c, ctypes.cast(buf, ctypes.c_void_p)))
            uid = torch.frombuffer(bytearray(buf), dtype=torch.uint8).clone()
        uid = uid.to(dev)
        dist.broadcast(uid, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        buf = (ctypes.c_uint8 * 128)(*uid.cpu().tolist())
        dp = ctypes.c_void_p()
        _lib.check(_lib.lib.dcll_dp_create(lib_c, ctypes.cast(buf, ctypes.c_void_p), dist.get_rank(group),
                                           dist.get_world_size(group), int(max_ctas), ctypes.byref(dp)))
        _DP_HANDLES[key] = dp
        return dp

    def learn_window_dp(self, x, labels, group=None, max_ctas=None):
        """Data-parallel ``learn_window``: every rank holds identical weights and its own shard of the batch
        (samples are independent in the forward pass, the state and the read-outs; the only coupling is the
        mean over the batch in the local loss).  Each layer's local gradients (gW, gb and, on the output
        layer, gWout, gbout) live in one flat bucket that is averaged over ranks with a single NCCL
        all-reduce per layer per timestep; the collective of layer l overlaps the forward/backward of layers
        l+1.. and is only waited for right before layer l's next forward, where the identical Adam step is
        applied on every rank.  Equals the single-process run at the global batch up to summation order.

        With the NCCL backend the whole window runs inside the C driver (``dcll_net_window_dp``: raw ncclAllReduce on a
        side stream, no per-timestep Python); other backends (gloo in the CPU tests) take the per-layer Python loop."""
        import torch.distributed as dist
        n = self.num_layers
        x_t, x_mode = (x.cells, _lib.X_CELLS) if isinstance(x, SpikeCells) else (_as_cuda_f32(x), _lib.X_DENSE)
        T, batch = int(x_t.shape[0]), int(x_t.shape[1])
        for s in self.dcll_slices:
            lay = s.dclllayer
            if lay.i2h.state.eps0.shape[0] != batch:
                import logging
                logging.warning("Batch size changed from {} to {} since last iteration. Reallocating states."
                                .format(lay.i2h.state.eps0.shape[0], batch))
                lay.i2h.init_state(batch, lay.im_dims)
            if _loss_kind(s.crit) == _lib.LOSS_EXTERNAL:
                raise NotImplementedError('learn_window_dp implements %s with default arguments' % ', '.join(NATIVE_LOSSES))
        rules = self._window_rules('learn_window_dp')
        win = self._window_buffers(batch)
        Layers, Trains = _lib.ConvLayer * n, _lib.TrainArgs * n
        layers, trains = Layers(), Trains()
        olds, states, buckets = [], [], []
        target = _as_cuda_f32(labels)
        t_stride = 0
        if target.dim() == 3:
            if target.shape[0] == T and T > 1:
                t_stride = target.shape[1] * target.shape[2]
            elif target.shape[0] != 1 and target.shape[0] != T:
                raise ValueError('labels [T,B,K] must cover the window: got %d rows for T = %d' % (target.shape[0], T))
        for i, s in enumerate(self.dcll_slices):
            lay = s.dclllayer
            old, _ = lay._fill_desc(layers[i], batch, x_mode if i == 0 else _lib.X_DENSE, win['outs'][i])
            olds.append(old)
            trains[i].loss_kind, trains[i].apply_update = _loss_kind(s.crit), 0
            trains[i].target = _lib.ptr(target)
            states.append(self._fill_slice(i, trains[i], rules))
            flat, views = grad_bucket(lay, x_t.device)
            trains[i].grad_w, trains[i].grad_b = _lib.ptr(views[0]), _lib.ptr(views[1])
            if lay.output_layer:
                trains[i].grad_wout, trains[i].grad_bout = _lib.ptr(views[2]), _lib.ptr(views[3])
            buckets.append(flat)
        clout = torch.empty((T, n, batch), dtype=torch.int32, device=x_t.device)
        stream = _lib.current_stream()
        burnin = int(self.dcll_slices[0].burnin)
        if dist.get_backend(group) == 'nccl':
            if max_ctas is None:
                # measured on 2 B200s (128x128, B = 64 per GPU): 4 and 8 CTAs scale alike (0.969 / 0.967 of the 1-GPU step),
                # 2 starves the 50 MB output_ bucket (0.941); fewer CTAs = fewer SMs held back from the persistent kernels
                max_ctas = int(os.environ.get('DCLL_DP_MAX_CTAS', '4'))
            dp = self._dp_handle(group, max_ctas)
            iter0 = (ctypes.c_int32 * n)(*[int(s.iter) for s in self.dcll_slices])
            bptr = (ctypes.c_void_p * n)(*[_lib.ptr(b) for b in buckets])
            bn = (ctypes.c_size_t * n)(*[b.numel() for b in buckets])
            if rules is not None:
                _lib.check(_lib.lib.dcll_net_window_dp_opt(dp, layers, trains, rules, n, _lib.ptr(x_t), _lib.ptr(target), t_stride,
                                                           T, burnin, iter0, _lib.ptr(clout), bptr, bn, stream))
            else:
                _lib.check(_lib.lib.dcll_net_window_dp(dp, layers, trains, n, _lib.ptr(x_t), _lib.ptr(target), t_stride, T, burnin,
                                                       iter0, _lib.ptr(clout), bptr, bn, stream))
            # the side stream's last collective was waited for by the main stream inside the driver: the buckets may be freed
        else:
            self._learn_window_dp_python(layers, trains, buckets, x_t, target, t_stride, T, clout, group, stream, burnin, rules)
        for i, s in enumerate(self.dcll_slices):
            s.dclllayer.i2h._commit_state(*olds[i], flips=T)
            s.dclllayer._ctx = None
            first = max(0, int(s.burnin) - int(s.iter) - 1)
            if first < T:
                s.clout.extend(clout[first:, i, :])
            s.iter += T
            self._store_slice(i, trains[i], rules, states[i])
        return clout

    def _learn_window_dp_python(self, layers, trains, buckets, x_t, target, t_stride, T, clout, group, stream, burnin, rules=None):
        """The same schedule issued layer by layer from Python over torch.distributed (any backend)."""
        n = self.num_layers
        pending, needs_apply = [None] * n, [False] * n
        step_bwd, apply = _lib.lib.dcll_conv_step_bwd_update, _lib.lib.dcll_conv_apply_update
        apply_opt = _lib.lib.dcll_conv_apply_update_opt
        x_stride = x_t[0].numel() * x_t.element_size()
        x_base = x_t.data_ptr()
        iters = [int(s.iter) for s in self.dcll_slices]

        def finish(i):
            # a backward ran for layer i: wait for its collective (a completed blocking one returns no handle) and
            # apply the identical Adam step on every rank
            if needs_apply[i]:
                if pending[i] is not None:
                    pending[i].wait()
                    pending[i] = None
                if rules is None:
                    _lib.check(apply(ctypes.byref(layers[i]), ctypes.byref(trains[i]), stream))
                else:
                    _lib.check(apply_opt(ctypes.byref(layers[i]), ctypes.byref(trains[i]),
                                         ctypes.pointer(rules[2 * i]), stream))
                needs_apply[i] = False

        # between two tensor-core layers of equal geometry the next layer's trace update rides in this layer's convolution
        # epilogue, as in dcll_net_window (it depends on this layer's spikes only, not on the weights being reduced)
        chain = _lib.lib.dcll_conv_step_fwd_chain
        fuse = [i + 1 < n and bool(_lib.lib.dcll_conv_chain_fusable(ctypes.byref(layers[i]), ctypes.byref(layers[i + 1])))
                for i in range(n)]
        for t in range(T):
            for i in range(n):
                finish(i)
                trains[i].target = target.data_ptr() + t * t_stride * 4
                xin = x_base + t * x_stride if i == 0 else layers[i - 1].spikes
                _lib.check(chain(ctypes.byref(layers[i]), ctypes.byref(layers[i + 1]) if fuse[i] else None,
                                 1 if i > 0 and fuse[i - 1] else 0, xin, clout[t, i].data_ptr(), stream))
                iters[i] += 1
                if iters[i] >= burnin:
                    _lib.check(step_bwd(ctypes.byref(layers[i]), ctypes.byref(trains[i]), stream))
                    pending[i] = allreduce_mean(buckets[i], group=group, async_op=True)
                    needs_apply[i] = True
        for i in range(n):
            finish(i)

    def learn_window(self, x, labels):
        """``for t in range(T): self.learn(x[t], labels[t])`` (train.py:249-251) in one call."""
        return self._run_window(x, labels, True)

    def test_window(self, x):
        """``for t in range(T): self.test(x[t])`` (test_radio_ml.py:144-145) in one call.  The radio_ml_conv stack on a
        16x16 plane in 'bf16x3' or 'f16x2' mode, quantised or not, with cell input takes the multi-timestep kernel (state on
        chip across timesteps), in the operand form of the per-timestep kernels of that mode."""
        if self._stack16_ok(x):
            return self._run_stack16(x)
        return self._run_window(x, None, False)

    # -- multi-timestep inference kernel (dcll_infer_stack16) -----------------------------------------
    def _stack16_ok(self, x):
        if not isinstance(x, SpikeCells) or self.num_layers != 3 or x.cells.dim() != 3:
            return False
        for i, s in enumerate(self.dcll_slices):
            lay, i2h = s.dclllayer, s.dclllayer.i2h
            if (tuple(int(v) for v in lay.im_dims) != (16, 16) or i2h.kernel_size != (7, 7) or i2h.padding != (3, 3)
                    or tuple(lay.pooling) != (1, 1) or i2h.out_channels != 32 or i2h.in_channels != (1 if i == 0 else 32)
                    or i2h.precision not in ('bf16x3', 'f16x2') or i2h.state.eps0.shape[0] != x.cells.shape[1]):
                return False
        # one kernel instantiation runs both 32 -> 32 layers: same operand form
        mode = self.dcll_slices[1].dclllayer.i2h.precision
        if mode != self.dcll_slices[2].dclllayer.i2h.precision:
            return False
        # f16x2: faster than the per-timestep f16x2 kernels up to B = 4096 (B200, T = 256), slower at B = 65536, where the pv
        # buffer holds one timestep per launch (DESIGN §4.5); larger batches keep the per-timestep kernels
        return mode != 'f16x2' or x.cells.shape[1] <= STACK16_F16X2_MAX_BATCH

    def _run_stack16(self, x, chunk=None):
        n, cells = 3, x.cells
        T, batch = int(cells.shape[0]), int(cells.shape[1])
        dev = cells.device
        win = self._window_buffers(batch)
        Layers = _lib.ConvLayer * n
        layers = Layers()
        for i, s in enumerate(self.dcll_slices):
            s.dclllayer._fill_desc(layers[i], batch, _lib.X_CELLS if i == 0 else _lib.X_DENSE, win['outs'][i])
            if layers[i].coef_mode == _lib.COEF_ELEMENT:
                return self._run_window(x, None, False)
        fsz = 32 * 256
        tc_max = chunk or max(1, min(16, T, int(3e9 // (3 * batch * fsz * 4))))
        key = ('stack16', batch, tc_max, dev)
        if getattr(self, '_s16', None) is None or self._s16['key'] != key:
            rows = tc_max * batch
            bufs = dict(key=key, pv=[torch.empty((rows, fsz), device=dev) for _ in range(n)], descs=[], keep=[])
            for i, s in enumerate(self.dcll_slices):
                lay = s.dclllayer
                d = _lib.ConvLayer()
                ctypes.memmove(ctypes.byref(d), ctypes.byref(layers[i]), ctypes.sizeof(d))
                d.B = rows
                po = torch.empty((rows, lay.target_size), device=dev)
                out = torch.empty((rows, lay.target_size), device=dev) if lay.output_layer else None
                d.pv, d.pvoutput, d.output = _lib.ptr(bufs['pv'][i]), _lib.ptr(po), _lib.ptr(out)
                ws = torch.empty(_lib.lib.dcll_conv_workspace_bytes(ctypes.byref(d)), dtype=torch.uint8, device=dev)
                d.workspace, d.workspace_bytes = _lib.ptr(ws), ws.numel()
                bufs['descs'].append(d)
                bufs['keep'] += [po, out, ws]
            bufs['clrows'] = torch.empty(rows, dtype=torch.int32, device=dev)
            self._s16 = bufs
        s16 = self._s16
        for i in range(n):      # parameter pointers may have moved since the buffers were built
            d = s16['descs'][i]
            d.wo, d.bo, d.wout, d.bout = layers[i].wo, layers[i].bo, layers[i].wout, layers[i].bout
        pv_ptrs = (ctypes.c_void_p * n)(*[_lib.ptr(t) for t in s16['pv']])
        clout = torch.empty((T, n, batch), dtype=torch.int32, device=dev)
        stream = _lib.current_stream()
        for t0 in range(0, T, tc_max):
            tc = min(tc_max, T - t0)
            _lib.check(_lib.lib.dcll_infer_stack16(layers, n, cells[t0].data_ptr(), tc, pv_ptrs, stream))
            for i in range(n):
                d = s16['descs'][i]
                d.B = tc * batch
                _lib.check(_lib.lib.dcll_conv_readout_rows(ctypes.byref(d), _lib.ptr(s16['clrows']), stream))
                clout[t0:t0 + tc, i, :] = s16['clrows'][:tc * batch].view(tc, batch)
        for i, s in enumerate(self.dcll_slices):
            s.dclllayer._ctx = None
            s.clout.extend(clout[:, i, :])
            s.iter += T
        return clout
