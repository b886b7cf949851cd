"""Host-side mirror of the reference's ``dcll/pytorch_libdcll.py`` on top of libdcll_b200.

Same class names, constructor signatures, attribute names and ``state_dict`` keys as the
reference (SURVEY.md section 8b), so that ``networks.ConvNetwork``, ``train.py`` and saved
``.pth`` files interchange.  All arithmetic of the per-timestep layer step runs in the
hand-written sm_100a kernels behind the C ABI in ``include/dcll_b200.h``; PyTorch only owns
the device memory.  There is no CPU path: tensors must live on a CUDA device.

Reference lines cited as ``ref:`` are in /root/reference/dcll/pytorch_libdcll.py.
"""
import ctypes
import logging
import math
from collections import Counter, namedtuple

import numpy as np
import torch
import torch.nn as nn
import torch.optim as optim

from .. import _lib

logger = logging.getLogger(__name__)

device = 'cuda'  # ref:34 -- module global imported by train.py:10 and networks/__init__.py:7


def _dev():
    return torch.device(device)


def _pair(v):
    return (int(v), int(v)) if not hasattr(v, '__len__') else (int(v[0]), int(v[1]))


# ------------------------------------------------------------------------------------------------
# vote accuracy (ref:44-69)
# ------------------------------------------------------------------------------------------------
def get_predictions_by_vote(pvoutput, labels):
    """ref:44-56.  ``pvoutput``: per-timestep predictions (list of [B] arrays or a DeviceClout);
    ``labels``: [T', B, K] one-hot.  Most frequent entry per sample, first-seen wins ties."""
    if isinstance(pvoutput, DeviceClout):
        pred = pvoutput.vote(labels.shape[-1] if hasattr(labels, 'shape') else None)
    else:
        cols = np.array(pvoutput).T
        pred = np.empty(len(cols))
        for i, col in enumerate(cols):
            pred[i] = Counter(col.tolist()).most_common(1)[0][0]
    lab = labels.detach().cpu().numpy() if torch.is_tensor(labels) else np.asarray(labels)
    lab = lab.argmax(axis=2).T
    true = np.empty(len(lab))
    for i, col in enumerate(lab):
        true[i] = Counter(col.tolist()).most_common(1)[0][0]
    return pred, true


def accuracy_by_vote(pvoutput, labels):
    pred, true = get_predictions_by_vote(pvoutput, labels)
    return float(np.mean(pred == true))


def accuracy_by_mean(pvoutput, labels):
    return float(np.mean((np.array(pvoutput) == labels.argmax(2).cpu().numpy())))


def accuracy_by_mse(pvoutput, labels):
    return torch.sum((pvoutput - labels) ** 2).item()


class DeviceClout:
    """Per-timestep class predictions kept on the device (replaces the reference's python list of
    ``argmax(1).cpu().numpy()`` arrays, ref:726-728, which costs a device sync per layer per step).

    Behaves like that list for ``len``, iteration, indexing and ``np.array``; rows are copied to
    the host once, on first access.
    """

    def __init__(self):
        self._buf = None
        self._n = 0
        self._host = None

    def __len__(self):
        return self._n

    def _reserve(self, batch, extra):
        need = self._n + extra
        if self._buf is None or self._buf.shape[1] != batch:
            self._buf = torch.empty((max(need, 64), batch), dtype=torch.int32, device=_dev())
            self._n = 0
        elif self._buf.shape[0] < need:
            grown = torch.empty((max(need, 2 * self._buf.shape[0]), batch), dtype=torch.int32, device=_dev())
            grown[:self._n] = self._buf[:self._n]
            self._buf = grown

    def next_row(self, batch):
        """Device row the kernel writes this step's argmax into."""
        self._reserve(batch, 1)
        row = self._buf[self._n]
        self._n += 1
        self._host = None
        return row

    def extend(self, rows):
        """rows: device int32 [n, B]."""
        if rows.shape[0] == 0:
            return
        self._reserve(rows.shape[1], rows.shape[0])
        self._buf[self._n:self._n + rows.shape[0]] = rows
        self._n += rows.shape[0]
        self._host = None

    def device_rows(self):
        return self._buf[:self._n]

    def numpy(self):
        if self._host is None:
            self._host = (self._buf[:self._n].cpu().numpy().astype(np.int64) if self._n
                          else np.zeros((0, 0), dtype=np.int64))
        return self._host

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype)

    def __iter__(self):
        return iter(self.numpy())

    def __getitem__(self, i):
        return self.numpy()[i]

    def vote_device(self, num_classes=None):
        """Device-side majority vote (dcll_vote): int32 [B] on the device, no host sync."""
        rows = self.device_rows()
        k = int(num_classes) if num_classes else int(rows.max().item()) + 1
        pred = torch.empty(rows.shape[1], dtype=torch.int32, device=rows.device)
        _lib.check(_lib.lib.dcll_vote(_lib.ptr(rows), rows.shape[0], rows.shape[1], rows.shape[1], k,
                                      _lib.ptr(pred), _lib.current_stream()))
        return pred

    def vote(self, num_classes=None):
        """Majority vote as a float numpy array like ref:47."""
        if self._n == 0:
            return np.empty(0)
        return self.vote_device(num_classes).cpu().numpy().astype(np.float64)


# ------------------------------------------------------------------------------------------------
# helpers shared by the conv core and the layer
# ------------------------------------------------------------------------------------------------
def _as_cuda_f32(t):
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    if t.device.type != 'cuda':
        t = t.to(_dev())
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class SpikeCells:
    """Compact layer-0 input: int32 [B, 2] (row, col) of the single spike of each sample's frame,
    as produced by ``data.utils.iq2spiketrain(..., as_cells=True)``.  Feeding it instead of the
    dense one-hot frame skips materialising [T,B,1,H,W] (8.6 GB at 128x128, T=1024)."""

    def __init__(self, cells, height, width):
        self.cells, self.height, self.width = cells, int(height), int(width)

    @property
    def shape(self):
        return torch.Size([self.cells.shape[0], 1, self.height, self.width])

    def dense(self):
        b = self.cells.shape[0]
        out = torch.empty((1, b, 1, self.height, self.width), dtype=torch.float32, device=self.cells.device)
        _lib.check(_lib.lib.dcll_cells_to_frames(_lib.ptr(self.cells), 1, b, self.height, self.width, _lib.ptr(out),
                                                 _lib.current_stream()))
        return out[0]


class _CoefView:
    """Time constants as the kernels want them.  The reference stores alpha/alphas/tau_m__dt/tau_s__dt
    as (1,) tensors or, with random_tau, as (Cin,H,W) tensors that hold ONE value per input channel
    (ref:391-405).  Per-channel planes are detected (once per parameter version) and passed as [Cin]
    vectors; genuinely per-element tensors (e.g. loaded from a foreign state_dict) are passed as is."""

    def __init__(self):
        self._key = None
        self.mode = _lib.COEF_SCALAR
        self.tensors = None

    def get(self, mod, cin, h, w):
        ps = (mod.alpha, mod.alphas, mod.tau_m__dt, mod.tau_s__dt)
        key = tuple((p.data_ptr(), p._version, tuple(p.shape)) for p in ps) + (cin, h, w)
        if key == self._key:
            return self.mode, self.tensors
        ts = [_as_cuda_f32(p.detach()) for p in ps]
        if all(t.numel() == 1 for t in ts):
            mode = _lib.COEF_SCALAR
        else:
            full = [t.expand(cin, h, w) if t.numel() == 1 else t for t in ts]
            for t in full:
                if tuple(t.shape) != (cin, h, w):
                    raise ValueError("time-constant tensor of shape %s does not match input (%d,%d,%d)"
                                     % (tuple(t.shape), cin, h, w))
            if all(bool((t == t[:, :1, :1]).all()) for t in full):
                mode, ts = _lib.COEF_CHANNEL, [t[:, 0, 0].contiguous() for t in full]
            else:
                mode, ts = _lib.COEF_ELEMENT, [t.contiguous() for t in full]
        self._key, self.mode, self.tensors = key, mode, ts
        return mode, ts


# ------------------------------------------------------------------------------------------------
# ContinuousConv2D / ContinuousRelativeRefractoryConv2D  (ref:296-509)
# ------------------------------------------------------------------------------------------------
class ContinuousConv2D(nn.Module):
    NeuronState = namedtuple('NeuronState', ('eps0', 'eps1'))

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=2, dilation=1, groups=1,
                 bias=True, alpha=.95, alphas=.9, act=nn.Sigmoid(), random_tau=False, spiking=True, **kwargs):
        super(ContinuousConv2D, self).__init__()
        if in_channels % groups != 0:                                   # ref:316-319
            raise ValueError('in_channels must be divisible by groups')
        if out_channels % groups != 0:
            raise ValueError('out_channels must be divisible by groups')
        if not (stride == 1 and dilation == 1 and groups == 1 and bias):
            raise NotImplementedError('libdcll_b200 implements stride=1, dilation=1, groups=1, bias=True '
                                      '(every shipped network spec); got stride=%r dilation=%r groups=%r bias=%r'
                                      % (stride, dilation, groups, bias))
        if not isinstance(act, nn.Sigmoid):
            raise NotImplementedError('only nn.Sigmoid() is implemented as local activation (ref: train.py:179)')
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.padding = _pair(kernel_size), _pair(padding)
        self.stride, self.dilation, self.groups = stride, dilation, groups
        self.random_tau, self.act, self.spiking = random_tau, act, spiking
        if not spiking:
            raise NotImplementedError('non-spiking layers are not implemented (every entry point uses spiking=True, '
                                      'networks/__init__.py:142)')
        # same torch-RNG consumption order as ref:342-356: weight, bias, then the four time constants
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels // groups, *self.kernel_size))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()
        self.alpha = nn.Parameter(torch.Tensor([alpha]), requires_grad=False)
        self.tau_m__dt = nn.Parameter(torch.Tensor([1. / (1 - self.alpha)]), requires_grad=False)
        self.alphas = nn.Parameter(torch.Tensor([alphas]), requires_grad=False)
        self.tau_s__dt = nn.Parameter(torch.Tensor([1. / (1 - self.alphas)]), requires_grad=False)
        self._coef = _CoefView()
        self._wt = None            # [Cin, KH*KW, CoutPad] kernel-side weight copy
        self._wt_key = None
        self._spare = None         # the other half of the ping-pong state
        self.quantized = False     # see quant.py
        self.precision = 'fp32'    # 'fp32' (parity mode), 'bf16x3' or 'f16x2' (tcgen05 tensor cores, where instantiated)
        self._wmma = None          # bf16 {hi,lo} weights in the tcgen05 B-operand layout
        self._wexp = None          # 'f16x2': device int32[4], exponent bookkeeping of the fp16 weight image (library-owned)
        self._aexp = None          # 'f16x2': (key, exponent) of the trace image scale
        self._e1mma = None         # bf16 {hi,lo} image of eps1 in the tcgen05 A-operand layout (written by the forward)

    # ref:359-366
    def reset_parameters(self):
        n = self.in_channels * self.kernel_size[0] * self.kernel_size[1]
        stdv = 1. / math.sqrt(n) / 250
        self.weight.data.uniform_(-stdv * 1e-2, stdv * 1e-2)
        self.bias.data.uniform_(-stdv, stdv)

    # ref:368-375
    def get_output_shape(self, im_dims):
        h = (im_dims[0] + 2 * self.padding[0] - self.dilation * (self.kernel_size[0] - 1) - 1) // self.stride + 1
        w = (im_dims[1] + 2 * self.padding[1] - self.dilation * (self.kernel_size[1] - 1) - 1) // self.stride + 1
        return h, w

    def _zeros_state(self, batch_size, im_dims, init_value):
        shape = [batch_size, self.in_channels, int(im_dims[0]), int(im_dims[1])]
        return torch.zeros(shape, device=_dev()) + init_value

    # ref:377-389 -- the non-refractory core randomises its time constants once
    def init_state(self, batch_size, im_dims, init_value=0):
        self.state = self.NeuronState(eps0=self._zeros_state(batch_size, im_dims, init_value),
                                      eps1=self._zeros_state(batch_size, im_dims, init_value))
        self._spare = None
        if self.random_tau:
            self.randomize_tau(im_dims)
            self.random_tau = False
        return self.state

    # ref:391-405 -- numpy RNG, tau_m drawn before tau_s
    def randomize_tau(self, im_dims, low=[5, 5], high=[10, 35]):
        taum = np.random.uniform(low[1], high[1], size=[self.in_channels]) * 1e-3
        taus = np.random.uniform(low[0], high[0], size=[self.in_channels]) * 1e-3
        shape = (int(im_dims[0]), int(im_dims[1]), self.in_channels)
        taum = np.broadcast_to(taum, shape).transpose(2, 0, 1)
        taus = np.broadcast_to(taus, shape).transpose(2, 0, 1)
        self.alpha = nn.Parameter(torch.Tensor(1 - 1e-3 / taum).to(_dev()), requires_grad=False)
        self.tau_m__dt = nn.Parameter(1. / (1 - self.alpha), requires_grad=False)
        self.alphas = nn.Parameter(torch.Tensor(1 - 1e-3 / taus).to(_dev()), requires_grad=False)
        self.tau_s__dt = nn.Parameter(1. / (1 - self.alphas), requires_grad=False)

    def init_prev(self, batch_size, im_dims):
        return torch.zeros(batch_size, self.in_channels, im_dims[0], im_dims[1])

    # -- kernel plumbing ----------------------------------------------------------------------
    wrp = 0.0
    alpharp = 0.65

    def _arp(self):
        return None

    def _check_batch(self, x):
        """ref:410-413 -- a batch-size change is a warning plus a fresh zero state, not an error."""
        st = self.state
        if not (x.shape[0] == st.eps0.shape[0] == st.eps1.shape[0]):
            logging.warning("Batch size changed from {} to {} since last iteration. Reallocating states."
                            .format(st.eps0.shape[0], x.shape[0]))
            self.init_state(x.shape[0], x.shape[2:4])

    def _sync_weight_t(self, desc):
        """Kernel-side weight copies: weight_t [Cin*KH*KW, CoutPad] (+ a dense dequantised copy behind it in
        quantised mode) and, for the tensor-core kernels, weight_mma.  Refreshed by the library after its own Adam
        steps; refreshed here when Python changed the parameter (load_state_dict, foreign optimiser, mode switch)."""
        w = self.weight
        key = (w.data_ptr(), w._version, self.quantized, self.precision)
        cout_pad = (self.out_channels + 31) // 32 * 32
        cinkk = self.in_channels * self.kernel_size[0] * self.kernel_size[1]
        n = cinkk * cout_pad + w.numel()
        if self._wt is None or self._wt.numel() != n or self._wt.device != w.device:
            self._wt = torch.zeros(n, dtype=torch.float32, device=w.device)
            self._wt_key = None
        desc.weight_t = _lib.ptr(self._wt)
        desc.quantized = 1 if self.quantized else 0
        if self.tensor_core_ok():
            n_mma = max(2 * self.weight.numel(), 4096)     # single input channel: [4 row pairs][2][2][32][8]
            if self._wmma is None or self._wmma.numel() != n_mma or self._wmma.device != w.device:
                self._wmma = torch.empty(n_mma, dtype=torch.bfloat16, device=w.device)
                self._wt_key = None
            desc.weight_mma = _lib.ptr(self._wmma)
        if self._wt_key != key:
            _lib.check(_lib.lib.dcll_conv_sync_weights(ctypes.byref(desc), _lib.current_stream()))
            self._wt_key = key

    def tensor_core_ok(self):
        """True when this core runs on the tcgen05 split-bf16 kernels (precision 'bf16x3' and an instantiated
        shape: 7x7, {1, 32} -> 32 channels; the layer additionally needs pooling 1, checked by the library).
        Other shapes stay on the FP32 FMA kernel."""
        if not (self.precision in ('bf16x3', 'f16x2') and self.kernel_size == (7, 7) and self.out_channels == 32):
            return False
        # single input channel: the operand pieces hold the column shifts x-padW .. x-padW+7 of the W input columns,
        # which covers every tap only while the output is not wider than the input (tc_supported, conv_fwd_tc.cu)
        return self.in_channels == 32 or (self.in_channels == 1 and 0 <= self.padding[1] <= 3)

    def f16_ok(self, height, width):
        """'f16x2' needs 32 input channels and the geometry of the row-pair weight-gradient kernel (even conv height, conv
        width a multiple of 8); other tensor-core layers of the network keep the split-bf16 kernels."""
        hc, wc = self.get_output_shape((height, width))
        return self.tensor_core_ok() and self.in_channels == 32 and hc % 2 == 0 and wc % 8 == 0

    def _trace_exp(self):
        """Exponent of the trace image: eps1 <= tau_s/(1-alphas) * tau_m/(1-alpha) for spike input (ref:415-416), and
        2^a_exp times that bound stays below 2^15 (fp16 maximum 65504).  One host read per parameter version."""
        ps = (self.alpha, self.alphas, self.tau_m__dt, self.tau_s__dt)
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if self._aexp is None or self._aexp[0] != key:
            a, als, tm, ts = (p.detach().double().flatten() for p in ps)
            bound = float(((ts / (1 - als)).max() * (tm / (1 - a)).max()).item())
            if not (bound > 0 and math.isfinite(bound)):
                raise ValueError("f16x2: time constants give no finite bound on eps1 (alpha, alphas must be < 1)")
            self._aexp = (key, int(math.floor(math.log2(32768.0 / bound))))
        return self._aexp[1]

    def _fill_core(self, desc, batch, height, width, x_mode):
        """Geometry, parameters and state pointers of the i2h core."""
        if self.weight.device.type != 'cuda':
            raise RuntimeError("libdcll_b200 has no CPU path: move the module to a CUDA device (.to('cuda'))")
        for p in (self.weight, self.bias):
            if not p.is_contiguous() or p.dtype != torch.float32:
                raise ValueError('weight/bias must be contiguous float32')
        desc.B, desc.Cin, desc.H, desc.W = batch, self.in_channels, height, width
        desc.Cout, desc.KH, desc.KW = self.out_channels, self.kernel_size[0], self.kernel_size[1]
        desc.padH, desc.padW = self.padding
        desc.x_mode = x_mode
        # 'bf16x3' selects the tensor-core kernels wherever the library has an instantiation for the shape
        # (forward: 7x7, 32->32; weight gradient: 7x7, {1,32}->32); other kernels of the layer stay FP32.
        desc.precision = {'bf16x3': _lib.PREC_BF16X3, 'f16x2': _lib.PREC_F16X2}.get(self.precision, _lib.PREC_FP32)
        if self.precision == 'f16x2':
            if self.f16_ok(height, width):
                if self._wexp is None or self._wexp.device != self.weight.device:
                    self._wexp = torch.zeros(4, dtype=torch.int32, device=self.weight.device)
                    self._wt_key = None                      # the image and its exponent are (re)built by the next sync
                desc.w_exp = _lib.ptr(self._wexp)
                desc.a_exp = self._trace_exp()
            else:
                desc.precision = _lib.PREC_BF16X3             # shapes without the fp16 kernels keep the split-bf16 form
        desc.alpharp, desc.wrp = float(self.alpharp), float(self.wrp)
        mode, ts = self._coef.get(self, self.in_channels, height, width)
        desc.coef_mode = mode
        desc.alpha, desc.alphas, desc.tau_m, desc.tau_s = (_lib.ptr(t) for t in ts)
        desc.weight, desc.bias = _lib.ptr(self.weight.data), _lib.ptr(self.bias.data)
        self._sync_weight_t(desc)
        st = self.state
        e0, e1 = st.eps0, st.eps1
        if not (e0.is_cuda and e0.is_contiguous() and e0.dtype == torch.float32):
            e0 = _as_cuda_f32(e0)
        if not (e1.is_cuda and e1.is_contiguous() and e1.dtype == torch.float32):
            e1 = _as_cuda_f32(e1)
        if (self._spare is None or self._spare[0].shape != e0.shape or self._spare[0].data_ptr() == e0.data_ptr()
                or self._spare[1].data_ptr() == e1.data_ptr()):
            self._spare = (torch.empty_like(e0), torch.empty_like(e1))
        desc.eps0[0], desc.eps0[1] = _lib.ptr(e0), _lib.ptr(self._spare[0])
        desc.eps1[0], desc.eps1[1] = _lib.ptr(e1), _lib.ptr(self._spare[1])
        desc.cur = 0
        if self.tensor_core_ok():
            # 16 bytes per position and group of 8 channels (a single channel fills the 8 slots with column shifts)
            n_img = 2 * e1.numel() // self.in_channels * max(self.in_channels, 8)
            if self._e1mma is None or self._e1mma.numel() != n_img or self._e1mma.device != e1.device:
                self._e1mma = torch.empty(n_img, dtype=torch.bfloat16, device=e1.device)
            desc.eps1_mma = _lib.ptr(self._e1mma)
        arp = self._arp()
        desc.arp = _lib.ptr(arp) if arp is not None else None
        return e0, e1, arp

    def _commit_state(self, old0, old1, arp, flips=1):
        """After `flips` kernel steps the new traces live in the spare pair iff flips is odd."""
        if flips % 2 == 1:
            new0, new1 = self._spare
            self._spare = (old0, old1)
        else:
            new0, new1 = old0, old1
        self.state = self.NeuronState(new0, new1) if arp is None else self.NeuronState(new0, new1, arp)

    def forward(self, input):
        """ref:407-426 -- returns (output, pv, pvmem) on the un-pooled conv grid."""
        dense = not isinstance(input, SpikeCells)
        x = _as_cuda_f32(input) if dense else input.cells
        shape = input.shape
        if shape[0] != self.state.eps0.shape[0]:
            self._check_batch(torch.empty(shape[0], 0, shape[2], shape[3]))
        batch, height, width = int(shape[0]), int(shape[2]), int(shape[3])
        desc = _lib.ConvLayer()
        old = self._fill_core(desc, batch, height, width, _lib.X_DENSE if dense else _lib.X_CELLS)
        hc, wc = self.get_output_shape((height, width))
        out_shape = (batch, self.out_channels, hc, wc)
        spikes, pv, pvmem = (torch.empty(out_shape, device=x.device) for _ in range(3))
        desc.poolH = desc.poolW = 1
        desc.K = 1
        desc.write_pvmem = 1
        desc.spikes, desc.pv, desc.pvmem = _lib.ptr(spikes), _lib.ptr(pv), _lib.ptr(pvmem)
        _lib.check(_lib.lib.dcll_conv_core_fwd(ctypes.byref(desc), _lib.ptr(x), _lib.current_stream()))
        self._commit_state(*old)
        return spikes, pv, pvmem


class ContinuousRelativeRefractoryConv2D(ContinuousConv2D):
    NeuronState = namedtuple('NeuronState', ('eps0', 'eps1', 'arp'))

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=2, dilation=1, groups=1,
                 bias=True, alpha=.95, alphas=.9, alpharp=.65, wrp=1, act=nn.Sigmoid(), random_tau=False, **kwargs):
        """Continuous local learning with relative refractory period (ref:435-466).
        *wrp*: weight of the relative refractory period."""
        super(ContinuousRelativeRefractoryConv2D, self).__init__(
            in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, alpha, alphas, act)
        self.wrp = wrp
        self.alpharp = alpharp
        self.tau_rp__dt = 1. / (1 - self.alpharp)
        self.iter = 0
        self.tau_set = False
        self.random_tau = random_tau

    # ref:468-483 -- quirk kept: the refractory core re-randomises tau on EVERY init_state
    def init_state(self, batch_size, im_dims, init_value=0):
        out_shape = [batch_size, self.out_channels] + list(self.get_output_shape(im_dims))
        self.state = self.NeuronState(eps0=self._zeros_state(batch_size, im_dims, init_value),
                                      eps1=self._zeros_state(batch_size, im_dims, init_value),
                                      arp=torch.zeros(out_shape, device=_dev()))
        self._spare = None
        if self.random_tau:
            self.randomize_tau(im_dims)
            self.random_tau = True
        return self.state

    def _arp(self):
        arp = self.state.arp
        if not (arp.is_cuda and arp.is_contiguous() and arp.dtype == torch.float32):
            arp = _as_cuda_f32(arp)
        return arp

    def forward(self, input):
        """ref:485-509 -- returns (output, pv, outpvmem)."""
        if not self.spiking:
            raise Exception('Refractory not allowed in non-spiking mode')
        return super(ContinuousRelativeRefractoryConv2D, self).forward(input)


# ------------------------------------------------------------------------------------------------
# Conv2dDCLLlayer  (ref:512-612)
# ------------------------------------------------------------------------------------------------
class Conv2dDCLLlayer(nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size=5, im_dims=(28, 28), target_size=10, pooling=None,
                 stride=1, dilation=1, padding=2, alpha=.95, alphas=.9, alpharp=.65, wrp=0, act=nn.Sigmoid(),
                 lc_dropout=False, lc_ampl=.5, spiking=True, random_tau=False, output_layer=False):
        super(Conv2dDCLLlayer, self).__init__()
        self.im_dims = im_dims
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lc_ampl = lc_ampl
        self.output_layer = output_layer
        if pooling is not None:                                         # ref:542-552
            pooling = _pair(pooling)
            self.pooling = pooling
            self.pool = nn.MaxPool2d(kernel_size=pooling, stride=pooling,
                                     padding=((pooling[0] - 1) // 2, (pooling[1] - 1) // 2))
        else:
            self.pooling = (1, 1)
            self.pool = lambda x: x
        if max(self.pooling) > 2 or min(self.pooling) < 1:
            raise NotImplementedError('libdcll_b200 implements pooling 1 or 2 per axis (all shipped specs); got %r'
                                      % (self.pooling,))
        self.kernel_size = kernel_size
        self.target_size = target_size
        if wrp > 0:                                                     # ref:555-563
            if not spiking:
                raise Exception('Non-spiking not allowed with refractory neurons')
            self.i2h = ContinuousRelativeRefractoryConv2D(
                in_channels, out_channels, kernel_size, padding=padding, dilation=dilation, stride=stride,
                alpha=alpha, alphas=alphas, alpharp=alpharp, wrp=wrp, act=act, random_tau=random_tau)
        else:
            self.i2h = ContinuousConv2D(in_channels, out_channels, kernel_size, padding=padding, dilation=dilation,
                                        stride=stride, alpha=alpha, alphas=alphas, act=act, spiking=spiking,
                                        random_tau=random_tau)
        conv_shape = self.i2h.get_output_shape(self.im_dims)
        # ref:567 derives the pooled shape by running the pool on zeros; for k = stride <= 2 that is H'//k
        self.output_shape = torch.Size([conv_shape[0] // self.pooling[0], conv_shape[1] // self.pooling[1]])
        if min(self.output_shape) < 1:
            raise RuntimeError('pooled output of %r is empty for im_dims %r' % (conv_shape, tuple(im_dims)))
        flat = int(np.prod(self.get_flat_size()))
        self.i2o = nn.Linear(flat, target_size, bias=True)              # ref:568-571, frozen
        self.i2o.weight.requires_grad = False
        self.i2o.bias.requires_grad = False
        if lc_dropout is not False:
            raise NotImplementedError('lc_dropout is not implemented (networks/__init__.py:143 passes False)')
        self.dropout = lambda x: x
        if output_layer:                                                # ref:577-579
            self.output_ = nn.Linear(flat, target_size, bias=True)
        self.reset_lc_parameters()
        self._workspace = None
        self._pool_idx = None
        self._g_u = None
        self._ctx = None

    def reset_lc_parameters(self):                                      # ref:583-587
        stdv = self.lc_ampl / math.sqrt(self.i2o.weight.size(1))
        self.i2o.weight.data.uniform_(-stdv, stdv)
        if self.i2o.bias is not None:
            self.i2o.bias.data.uniform_(-stdv, stdv)

    def get_flat_size(self):                                            # ref:589-591
        w, h = self.get_output_shape()
        return int(w * h * self.out_channels)

    def get_output_shape(self):                                         # ref:593-597
        conv_shape = self.i2h.get_output_shape(self.im_dims)
        return conv_shape[0] // self.pooling[0], conv_shape[1] // self.pooling[1]

    def init_hiddens(self, batch_size, init_value=0):                   # ref:610-612
        self.i2h.init_state(batch_size, self.im_dims, init_value=init_value)
        return self

    # -- kernel plumbing ----------------------------------------------------------------------
    def _fill_desc(self, desc, batch, x_mode, persistent_outputs):
        """Complete descriptor of this layer for `batch` samples; returns the objects to keep alive."""
        h, w = int(self.im_dims[0]), int(self.im_dims[1])
        old = self.i2h._fill_core(desc, batch, h, w, x_mode)
        dev = self.i2h.weight.device
        desc.poolH, desc.poolW = self.pooling
        desc.K = int(self.target_size)
        desc.output_layer = 1 if self.output_layer else 0
        for lin in [self.i2o] + ([self.output_] if self.output_layer else []):
            if lin.weight.device != dev or not lin.weight.is_contiguous():
                raise RuntimeError('read-out parameters must be contiguous and on the same device as i2h')
        desc.wo, desc.bo = _lib.ptr(self.i2o.weight.data), _lib.ptr(self.i2o.bias.data)
        if self.output_layer:
            desc.wout, desc.bout = _lib.ptr(self.output_.weight.data), _lib.ptr(self.output_.bias.data)
        hc, wc = self.i2h.get_output_shape((h, w))
        hp, wp = self.get_output_shape()
        pooled = (batch, self.out_channels, hp, wp)
        if max(self.pooling) > 1:
            if self._pool_idx is None or tuple(self._pool_idx.shape) != pooled or self._pool_idx.device != dev:
                self._pool_idx = torch.empty(pooled, dtype=torch.uint8, device=dev)
            desc.pool_idx = _lib.ptr(self._pool_idx)
        if persistent_outputs is None:
            outs = dict(spikes=torch.empty(pooled, device=dev), pv=torch.empty(pooled, device=dev),
                        pvmem=torch.empty((batch, self.out_channels, hc, wc), device=dev),
                        pvoutput=torch.empty((batch, self.target_size), device=dev),
                        output=torch.empty((batch, self.target_size), device=dev) if self.output_layer else None)
            desc.write_pvmem = 1
        else:
            outs = persistent_outputs
            desc.write_pvmem = 1 if outs.get('pvmem') is not None else 0
        desc.spikes, desc.pv, desc.pvoutput = _lib.ptr(outs['spikes']), _lib.ptr(outs['pv']), _lib.ptr(outs['pvoutput'])
        desc.pvmem = _lib.ptr(outs.get('pvmem'))
        desc.output = _lib.ptr(outs.get('output'))
        if self._g_u is None or tuple(self._g_u.shape) != pooled or self._g_u.device != dev:
            self._g_u = torch.empty(pooled, device=dev)
        desc.g_u = _lib.ptr(self._g_u)
        if desc.precision == _lib.PREC_F16X2:
            desc.g_exp = self._grad_exp(batch)
        need = _lib.lib.dcll_conv_workspace_bytes(ctypes.byref(desc))
        if self._workspace is None or self._workspace.numel() < need or self._workspace.device != dev:
            self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        desc.workspace, desc.workspace_bytes = _lib.ptr(self._workspace), self._workspace.numel()
        return old, outs

    def _grad_exp(self, batch):
        """Exponent of the g_u image ('f16x2'): |g_u| <= sum_k |g_o| |Wo| / 4 <= max|Wo| / (4 B) whenever sum_k |g_o| <= 1/B per
        row: the mean-reduced SmoothL1 / Huber / L1 / BCE-with-logits / soft-margin / hinge losses (|g_o| <= 1/(B K)) and
        KL divergence against targets in [0, 1].  2^4 of slack covers cross-entropy (sum_k |g_o| <= 2/B for probability
        targets), MSE residuals above 1 and external losses; MSE and Poisson NLL are unbounded, and the store saturates
        beyond the slack.  One host read per version of the frozen read-out."""
        w = self.i2o.weight
        key = (w.data_ptr(), w._version, batch)
        if getattr(self, '_gexp', None) is None or self._gexp[0] != key:
            bound = float(w.detach().abs().max().item()) / (4.0 * batch) * 16.0
            self._gexp = (key, int(math.floor(math.log2(16384.0 / bound))) if bound > 0 else 0)
        return self._gexp[1]

    def _input(self, input):
        if isinstance(input, SpikeCells):
            if self.in_channels != 1:
                raise ValueError('SpikeCells input needs in_channels == 1')
            return input.cells, _lib.X_CELLS, int(input.cells.shape[0])
        x = _as_cuda_f32(input)
        if x.dim() != 4 or x.shape[1] != self.in_channels or tuple(x.shape[2:4]) != tuple(int(v) for v in self.im_dims):
            raise ValueError('expected input [B,%d,%d,%d], got %s' % (self.in_channels, self.im_dims[0],
                                                                       self.im_dims[1], tuple(x.shape)))
        return x, _lib.X_DENSE, int(x.shape[0])

    def forward(self, input, clout_row=None):
        """ref:599-608 -> (output, pvoutput, pv, pvmem); `output` is the pooled spike tensor, or the
        logits of output_ on the output layer.  One fused launch sequence, no host sync."""
        x, x_mode, batch = self._input(input)
        if batch != self.i2h.state.eps0.shape[0]:
            self.i2h._check_batch(torch.empty(batch, 0, int(self.im_dims[0]), int(self.im_dims[1])))
        desc = _lib.ConvLayer()
        old, outs = self._fill_desc(desc, batch, x_mode, None)
        _lib.check(_lib.lib.dcll_conv_step_fwd(ctypes.byref(desc), _lib.ptr(x), _lib.ptr(clout_row),
                                               _lib.current_stream()))
        self.i2h._commit_state(*old)
        self._ctx = (desc, outs, x)
        output = outs['output'] if self.output_layer else outs['spikes']
        return output, outs['pvoutput'], outs['pv'], outs['pvmem']



# ------------------------------------------------------------------------------------------------
# Dense layers  (ref:72-274)
# ------------------------------------------------------------------------------------------------
class CLLDenseModule(nn.Module):
    NeuronState = namedtuple('NeuronState', ['eps0', 'eps1'])

    def __init__(self, in_channels, out_channels, bias=True, alpha=.9, alphas=.85, act=nn.Sigmoid(), spiking=True,
                 random_tau=False):
        super(CLLDenseModule, self).__init__()
        if not bias:
            raise NotImplementedError('bias=False is not implemented')
        if not isinstance(act, nn.Sigmoid) or not spiking:
            raise NotImplementedError('only spiking layers with nn.Sigmoid() are implemented')
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()
        self.act, self.random_tau, self.spiking = act, random_tau, spiking
        self.alpha = nn.Parameter(torch.Tensor([alpha]), requires_grad=False)          # ref:87-94
        self.tau_m__dt = nn.Parameter(torch.Tensor([1. / (1 - self.alpha)]), requires_grad=False)
        self.alphas = nn.Parameter(torch.Tensor([alphas]), requires_grad=False)
        self.tau_s__dt = nn.Parameter(torch.Tensor([1. / (1 - self.alphas)]), requires_grad=False)

    wrp = 0.0
    alpharp = 0.65

    def reset_parameters(self):                                         # ref:102-106
        stdv = 1. / math.sqrt(self.weight.size(1))
        self.weight.data.uniform_(-stdv * 1e-2, stdv * 1e-2)
        self.bias.data.uniform_(-stdv, stdv)

    def _zeros(self, batch_size, n, init_value):
        return torch.zeros(batch_size, n, device=_dev()) + init_value

    def init_state(self, batch_size, init_value=0):                     # ref:108-117 (re-randomises tau every time)
        self.state = self.NeuronState(eps0=self._zeros(batch_size, self.in_channels, init_value),
                                      eps1=self._zeros(batch_size, self.in_channels, init_value))
        if self.random_tau:
            self.randomize_tau()
        return self.state

    def randomize_tau(self, low=[5, 5], high=[10, 35]):                 # ref:119-129
        taum = np.random.uniform(low[1], high[1], size=[self.in_channels]) * 1e-3
        taus = np.random.uniform(low[0], high[0], size=[self.in_channels]) * 1e-3
        self.alpha = nn.Parameter(torch.Tensor(1 - 1e-3 / taum).to(_dev()), requires_grad=False)
        self.tau_m__dt = nn.Parameter(1. / (1 - self.alpha), requires_grad=False)
        self.alphas = nn.Parameter(torch.Tensor(1 - 1e-3 / taus).to(_dev()), requires_grad=False)
        self.tau_s__dt = nn.Parameter(1. / (1 - self.alphas), requires_grad=False)

    def _arp(self):
        return None

    def _step(self, input, wo, bo, clout_row=None):
        """Trace update + synapse + neuron (+ read-out when wo is given); returns the tensors and the descriptor."""
        if self.weight.device.type != 'cuda':
            raise RuntimeError("libdcll_b200 has no CPU path: move the module to a CUDA device (.to('cuda'))")
        x = _as_cuda_f32(input)
        if not (x.shape[0] == self.state.eps0.shape[0] == self.state.eps1.shape[0]):     # ref:134-137
            logger.warning("Batch size changed from {} to {} since last iteration. Reallocating states."
                           .format(self.state.eps0.shape[0], x.shape[0]))
            self.init_state(x.shape[0])
        batch, dev = int(x.shape[0]), x.device
        d = _lib.DenseLayer()
        d.B, d.In, d.Out = batch, self.in_channels, self.out_channels
        d.alpharp, d.wrp = float(self.alpharp), float(self.wrp)
        ts = [_as_cuda_f32(p.detach()) for p in (self.alpha, self.alphas, self.tau_m__dt, self.tau_s__dt)]
        if all(t.numel() == 1 for t in ts):
            d.coef_mode = _lib.COEF_SCALAR
        else:
            ts = [t.expand(self.in_channels).contiguous() if t.numel() == 1 else t.reshape(-1) for t in ts]
            d.coef_mode = _lib.COEF_CHANNEL
        d.alpha, d.alphas, d.tau_m, d.tau_s = (_lib.ptr(t) for t in ts)
        d.weight, d.bias = _lib.ptr(self.weight.data), _lib.ptr(self.bias.data)
        e0, e1 = _as_cuda_f32(self.state.eps0), _as_cuda_f32(self.state.eps1)
        d.eps0, d.eps1 = _lib.ptr(e0), _lib.ptr(e1)
        arp = self._arp()
        if arp is not None:
            arp = _as_cuda_f32(arp)
            d.arp = _lib.ptr(arp)
        k = int(wo.shape[0]) if wo is not None else 1
        d.K = k
        outs = dict(spikes=torch.empty((batch, self.out_channels), device=dev),
                    pv=torch.empty((batch, self.out_channels), device=dev),
                    vmem=torch.empty((batch, self.out_channels), device=dev),
                    pvoutput=torch.empty((batch, k), device=dev))
        if wo is None:      # stand-alone i2h call: a 1-row dummy read-out keeps the entry point uniform
            wo, bo = torch.zeros((1, self.out_channels), device=dev), torch.zeros(1, device=dev)
        d.wo, d.bo = _lib.ptr(wo), _lib.ptr(bo)
        d.spikes, d.pv, d.vmem, d.pvoutput = (_lib.ptr(outs[n]) for n in ('spikes', 'pv', 'vmem', 'pvoutput'))
        _lib.check(_lib.lib.dcll_dense_step_fwd(ctypes.byref(d), _lib.ptr(x), _lib.ptr(clout_row), _lib.current_stream()))
        self.state = self.NeuronState(e0, e1) if arp is None else self.NeuronState(e0, e1, arp)
        return outs, (d, ts, wo, bo, x)

    def forward(self, input):                                           # ref:131-148
        outs, _ = self._step(input, None, None)
        return outs['spikes'], outs['pv'], outs['vmem']


class CLLDenseRRPModule(CLLDenseModule):
    NeuronState = namedtuple('NeuronState', ('eps0', 'eps1', 'arp'))

    def __init__(self, in_channels, out_channels, bias=True, alpha=.95, alphas=.9, alpharp=.65, wrp=100,
                 act=nn.Sigmoid(), spiking=True, random_tau=False):
        super(CLLDenseRRPModule, self).__init__(in_channels, out_channels, bias, alpha, alphas, act, spiking=spiking,
                                                random_tau=random_tau)
        self.wrp = wrp
        self.alpharp = alpharp

    def init_state(self, batch_size, init_value=0):                     # ref:160-169 (no tau randomisation here)
        self.state = self.NeuronState(eps0=self._zeros(batch_size, self.in_channels, init_value),
                                      eps1=self._zeros(batch_size, self.in_channels, init_value),
                                      arp=self._zeros(batch_size, self.out_channels, init_value))
        return self.state

    def _arp(self):
        return self.state.arp

    def forward(self, input):                                           # ref:171-195
        if not self.spiking:
            raise Exception('Refractory not allowed in non-spiking mode')
        return super(CLLDenseRRPModule, self).forward(input)


class DenseDCLLlayer(nn.Module):
    def __init__(self, in_channels, out_channels, target_size=None, bias=True, alpha=.9, alphas=.85, alpharp=.65,
                 wrp=0., act=nn.Sigmoid(), lc_dropout=False, lc_ampl=.5, spiking=True, random_tau=False,
                 output_layer=False):
        if target_size is None:
            target_size = out_channels
        super(DenseDCLLlayer, self).__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lc_ampl = lc_ampl
        self.target_size = target_size
        self.output_layer = False                                       # ref:222 (hard-coded in the reference)
        if wrp > 0:
            self.i2h = CLLDenseRRPModule(in_channels, out_channels, alpha=alpha, alphas=alphas, alpharp=alpharp,
                                         wrp=wrp, bias=bias, act=act, spiking=spiking, random_tau=random_tau)
        else:
            self.i2h = CLLDenseModule(in_channels, out_channels, alpha=alpha, alphas=alphas, bias=bias, act=act,
                                      spiking=spiking, random_tau=random_tau)
        self.i2o = nn.Linear(out_channels, target_size, bias=bias)      # ref:229-232, frozen
        self.i2o.weight.requires_grad = False
        if bias:
            self.i2o.bias.requires_grad = False
        self.input_size = self.out_channels
        self.reset_lc_parameters()
        self.lc_dropout = lc_dropout
        if lc_dropout is not False:
            raise NotImplementedError('lc_dropout is not implemented')
        self.dropout = lambda x: x
        self._ctx = None

    def reset_lc_parameters(self):                                      # ref:244-248
        stdv = self.lc_ampl / math.sqrt(self.i2o.weight.size(1))
        self.i2o.weight.data.uniform_(-stdv, stdv)
        if self.i2o.bias is not None:
            self.i2o.bias.data.uniform_(-stdv, stdv)

    def forward(self, input, clout_row=None):                           # ref:250-255
        x = _as_cuda_f32(input).reshape(-1, self.in_channels)
        outs, ctx = self.i2h._step(x, self.i2o.weight.data, self.i2o.bias.data, clout_row)
        self._ctx = (ctx, outs)
        return outs['spikes'], outs['pvoutput'], outs['pv'], outs['vmem']

    def init_hiddens(self, batch_size, init_value=0):                   # ref:257-259
        self.i2h.init_state(batch_size, init_value=init_value)
        return self

    def reset_tracks(self, mask=None):                                  # ref:261-266 (the mask=None branch reads a
        if mask is None:                                                #  non-existent field in the reference; fixed)
            self.init_hiddens(self.i2h.state.eps0.shape[0])
            return
        for field in self.i2h.state:
            field[mask] = 0.

# ------------------------------------------------------------------------------------------------
# optimiser / loss adapters
# ------------------------------------------------------------------------------------------------
NATIVE_LOSSES = ('SmoothL1Loss', 'HuberLoss', 'MSELoss', 'L1Loss', 'CrossEntropyLoss', 'BCEWithLogitsLoss',
                 'MultiLabelSoftMarginLoss', 'SoftMarginLoss', 'KLDivLoss', 'PoissonNLLLoss', 'HingeEmbeddingLoss')


def _loss_kind(crit):
    """The device loss kind of a criterion: instances of exactly these torch.nn classes with their default arguments
    (NATIVE_LOSSES; mean reduction).  Anything else -- a subclass, other arguments -- is LOSS_EXTERNAL: the per-step API
    takes its gradient from autograd, the window drivers refuse it."""
    t = type(crit)
    if getattr(crit, 'reduction', None) != 'mean':
        return _lib.LOSS_EXTERNAL
    if (t is nn.SmoothL1Loss and getattr(crit, 'beta', 1.0) == 1.0) or (t is nn.HuberLoss and crit.delta == 1.0):
        return _lib.LOSS_SMOOTHL1
    if t is nn.MSELoss:
        return _lib.LOSS_MSE
    if t is nn.L1Loss:
        return _lib.LOSS_L1
    if t is nn.CrossEntropyLoss and crit.weight is None and crit.label_smoothing == 0.0 and crit.ignore_index == -100:
        return _lib.LOSS_CROSS_ENTROPY
    if (t is nn.BCEWithLogitsLoss and crit.weight is None and crit.pos_weight is None) or \
            (t is nn.MultiLabelSoftMarginLoss and crit.weight is None):
        return _lib.LOSS_BCE_LOGITS
    if t is nn.SoftMarginLoss:
        return _lib.LOSS_SOFT_MARGIN
    if t is nn.KLDivLoss and not crit.log_target:
        return _lib.LOSS_KL_DIV
    if t is nn.PoissonNLLLoss and crit.log_input and not crit.full:
        return _lib.LOSS_POISSON_NLL
    if t is nn.HingeEmbeddingLoss and crit.margin == 1.0:
        return _lib.LOSS_HINGE
    return _lib.LOSS_EXTERNAL


def _step_loss_kind(crit, target, pred):
    """_loss_kind for one per-step backward: the kinds added after the first three read the target as a [B,K] array like
    the read-out, so any other target form (class indices for CrossEntropyLoss, a broadcast) goes through autograd."""
    kind = _loss_kind(crit)
    if kind > _lib.LOSS_EXTERNAL and tuple(target.shape) != tuple(pred.shape):
        return _lib.LOSS_EXTERNAL
    return kind


def _is_plain_adam(opt):
    if type(opt) is not optim.Adam or len(opt.param_groups) != 1:
        return False
    g = opt.param_groups[0]
    return not (g.get('amsgrad') or g.get('maximize') or g.get('capturable') or g.get('differentiable')
                or g.get('decoupled_weight_decay'))


def _adam_state(opt, p):
    """optimizer.state[p] exactly as torch.optim.Adam lazily creates it, so state_dicts interchange."""
    st = opt.state[p]
    if len(st) == 0:
        st['step'] = torch.tensor(0.0, dtype=torch.float32)
        st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
    return st


def _fill_adam(adam, opt, pw, pb):
    g = opt.param_groups[0]
    adam.lr, (adam.beta1, adam.beta2) = float(g['lr']), (float(g['betas'][0]), float(g['betas'][1]))
    adam.eps, adam.weight_decay = float(g['eps']), float(g['weight_decay'])
    sw, sb = _adam_state(opt, pw), _adam_state(opt, pb)
    adam.step = int(sw['step'])
    adam.m_w, adam.v_w = _lib.ptr(sw['exp_avg']), _lib.ptr(sw['exp_avg_sq'])
    adam.m_b, adam.v_b = _lib.ptr(sb['exp_avg']), _lib.ptr(sb['exp_avg_sq'])
    return sw, sb


def _store_steps(states, step):
    for st in states:
        st['step'] = torch.tensor(float(step), dtype=torch.float32)


# optimizers the fused kernels apply (with the single-param-group, non-maximize, non-capturable, non-differentiable options
# _device_optim checks); any other optimizer takes torch's optimizer.step() in the per-step API
DEVICE_OPTIMIZERS = ('Adam', 'AdamW', 'Adamax', 'NAdam', 'RAdam')


def _device_optim(opt):
    """The update rule (_lib.OPT_ADAMW / OPT_ADAMAX / OPT_NADAM / OPT_RADAM) the fused kernels apply for `opt`, or None: exact
    torch.optim.AdamW (or Adam(decoupled_weight_decay=True)) without amsgrad, Adamax, NAdam or RAdam, with one param group,
    maximize, capturable and differentiable off and a float lr.  Plain Adam is _is_plain_adam's (None here)."""
    if len(opt.param_groups) != 1:
        return None
    g = opt.param_groups[0]
    if g.get('maximize') or g.get('capturable') or g.get('differentiable') or type(g.get('lr')) is not float:
        return None
    t = type(opt)
    if t is optim.AdamW or (t is optim.Adam and g.get('decoupled_weight_decay')):
        return None if g.get('amsgrad') else _lib.OPT_ADAMW
    return {optim.Adamax: _lib.OPT_ADAMAX, optim.NAdam: _lib.OPT_NADAM, optim.RAdam: _lib.OPT_RADAM}.get(t)


def _optim_state(opt, p, kind):
    """optimizer.state[p] exactly as the torch class of rule `kind` lazily creates it, so state_dicts interchange."""
    st = opt.state[p]
    if len(st) == 0:
        st['step'] = torch.tensor(0.0, dtype=torch.float32)
        if kind == _lib.OPT_NADAM:
            st['mu_product'] = torch.tensor(1.0, dtype=torch.float32)
        st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        st['exp_inf' if kind == _lib.OPT_ADAMAX else 'exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
    return st


def _fill_optim(adam, rule, opt, pw, pb):
    """dcll_adam + dcll_optim of a device optimizer (plain Adam: rule.kind = OPT_ADAM and _fill_adam); returns the states of
    the weight and the bias, which _store_optim updates after the call."""
    kind = _lib.OPT_ADAM if _is_plain_adam(opt) else _device_optim(opt)
    rule.kind = kind
    if kind == _lib.OPT_ADAM:
        return _fill_adam(adam, opt, pw, pb)
    g = opt.param_groups[0]
    adam.lr, (adam.beta1, adam.beta2) = float(g['lr']), (float(g['betas'][0]), float(g['betas'][1]))
    adam.eps, adam.weight_decay = float(g['eps']), float(g['weight_decay'])
    sw, sb = _optim_state(opt, pw, kind), _optim_state(opt, pb, kind)
    adam.step = int(sw['step'])
    v = 'exp_inf' if kind == _lib.OPT_ADAMAX else 'exp_avg_sq'
    adam.m_w, adam.v_w = _lib.ptr(sw['exp_avg']), _lib.ptr(sw[v])
    adam.m_b, adam.v_b = _lib.ptr(sb['exp_avg']), _lib.ptr(sb[v])
    rule.decoupled_wd = 1 if g.get('decoupled_weight_decay') else 0
    rule.momentum_decay = float(g.get('momentum_decay', 0.0))
    rule.mu_product = float(sw['mu_product']) if kind == _lib.OPT_NADAM else 1.0
    return sw, sb


def _store_optim(states, adam, rule):
    _store_steps(states, adam.step)
    if rule.kind == _lib.OPT_NADAM:
        for st in states:
            st['mu_product'] = torch.tensor(rule.mu_product, dtype=torch.float32)


def _on_device(*opts):
    """True when every optimizer is one the fused kernels apply (plain Adam or a _device_optim rule)."""
    return all(_is_plain_adam(o) or _device_optim(o) is not None for o in opts)


def _optims_of(s):
    lay = s.dclllayer
    return (s.optimizer, s.optimizer2) if lay.output_layer else (s.optimizer,)


# ------------------------------------------------------------------------------------------------
# DCLLBase / DCLLClassification  (ref:615-749)
# ------------------------------------------------------------------------------------------------
class DCLLBase(nn.Module):
    num_instances = 0

    def __init__(self, dclllayer, name='DCLLbase', batch_size=48, loss=torch.nn.MSELoss, optimizer=optim.SGD,
                 kwargs_optimizer={'lr': 5e-5}, burnin=200, collect_stats=False):
        """
        *dclllayer*: layer that supports local learning
        *batch_size*: used for initialization
        *loss*: torch loss class (None for inference-only slices, test_radio_ml.py:93-95)
        *optimizer*: torch optimizer class (None for inference-only slices)
        *kwargs_optimizer*: options passed to the optimizer
        *collect_stats*: whether activity statistics are collected during learning
        """
        super(DCLLBase, self).__init__()
        self.dclllayer = dclllayer
        if loss is not None:                                            # ref:629-632
            self.crit = loss().to(device)
            self.output_crit = loss().to(device)
        if optimizer is not None:                                       # ref:633-638
            self.optimizer = optimizer(dclllayer.i2h.parameters(), **kwargs_optimizer)
            if self.dclllayer.output_layer:
                self.optimizer2 = optimizer(dclllayer.output_.parameters(), lr=1e-4)
        self.burnin = burnin
        self.batch_size = batch_size
        self.collect_stats = collect_stats
        self.init(self.batch_size)
        self.stats_bins = np.linspace(0, 1, 20)
        self.name = name
        self.slice_id = DCLLBase.num_instances
        DCLLBase.num_instances += 1

    def init(self, batch_size, init_states=True):                       # ref:648-653
        self.clout = DeviceClout()
        self.activity_hist = []
        self.iter = 0
        if init_states:
            self.dclllayer.init_hiddens(batch_size, init_value=0)

    def _collect(self, pv):
        if self.collect_stats and (self.iter % 20) == 0:                # ref:658-661, histogram on the device
            h = torch.histc(pv.detach().float(), bins=len(self.stats_bins) - 1, min=0.0, max=1.0)
            self.activity_hist.append(h)

    def forward(self, input, clout_row=None):                           # ref:655-662
        self.iter += 1
        o, p, pv, pvmem = self.dclllayer.forward(input, clout_row)
        self._collect(pv)
        return o, p, pv, pvmem

    def write_stats(self, writer, label, epoch):                        # ref:664-688
        writer.add_histogram(self.name + '/weight', self.dclllayer.i2h.weight.flatten(), epoch)
        writer.add_histogram(self.name + '/bias', self.dclllayer.i2h.bias.flatten(), epoch)
        if self.collect_stats and len(self.activity_hist) > 0:
            pd = torch.stack(self.activity_hist).float().mean(0).cpu().numpy()
            pd = pd / pd.sum()
            writer.add_scalar(self.name + '/low_pv/' + label, pd[0], epoch)
            writer.add_scalar(self.name + '/high_pv/' + label, pd[-1], epoch)
            print(self.name + ' low:{0:1.3} high:{1:1.3}'.format(pd[0], pd[-1]))

    def _bwd_update(self, target, do_train):
        """Local gradient + optimiser step(s) for the forward pass that just ran (ref:693-714)."""
        lay = self.dclllayer
        if isinstance(lay, DenseDCLLlayer):
            return self._bwd_update_dense(target, do_train)
        desc, outs, _x = lay._ctx
        targ = _as_cuda_f32(target)
        args = _lib.TrainArgs()
        args.target = _lib.ptr(targ)
        keep = [targ]
        kind = _step_loss_kind(self.crit, targ, outs['pvoutput'])
        args.loss_kind = kind
        if kind == _lib.LOSS_EXTERNAL:
            # any other loss: its gradient w.r.t. the [B,K] read-outs comes from autograd
            pvo = outs['pvoutput'].detach().clone().requires_grad_(True)
            loss = self.crit(pvo, targ)
            if lay.output_layer:
                out = outs['output'].detach().clone().requires_grad_(True)
                loss = loss + self.output_crit(out, targ)
            loss.backward()
            keep += [pvo.grad, out.grad if lay.output_layer else None]
            args.g_o_ext = _lib.ptr(pvo.grad.contiguous())
            if lay.output_layer:
                args.g_o2_ext = _lib.ptr(out.grad.contiguous())
            loss_t = loss.detach().reshape(1)
        else:
            loss_t = torch.zeros(1, device=targ.device)
            args.loss_out = _lib.ptr(loss_t)
        fused = do_train and _is_plain_adam(self.optimizer) and \
            (not lay.output_layer or _is_plain_adam(self.optimizer2))
        # AdamW / Adamax / NAdam / RAdam (and plain Adam beside them) go through the _opt entry point
        rules = (_lib.Optim * 2)() if do_train and not fused and _on_device(*_optims_of(self)) else None
        i2h = lay.i2h
        states = []
        if rules is not None:
            args.apply_update = 1
            states.append(_fill_optim(args.adam_i2h, rules[0], self.optimizer, i2h.weight, i2h.bias))
            if lay.output_layer:
                states.append(_fill_optim(args.adam_out, rules[1], self.optimizer2, lay.output_.weight, lay.output_.bias))
        elif fused:
            args.apply_update = 1
            states.append(_fill_adam(args.adam_i2h, self.optimizer, i2h.weight, i2h.bias))
            if lay.output_layer:
                states.append(_fill_adam(args.adam_out, self.optimizer2, lay.output_.weight, lay.output_.bias))
        else:
            args.apply_update = 0
            params = [i2h.weight, i2h.bias] + ([lay.output_.weight, lay.output_.bias] if lay.output_layer else [])
            for p in params:
                if p.grad is None or p.grad.shape != p.shape or not p.grad.is_contiguous():
                    p.grad = torch.zeros_like(p)
            args.grad_w, args.grad_b = _lib.ptr(i2h.weight.grad), _lib.ptr(i2h.bias.grad)
            if lay.output_layer:
                args.grad_wout, args.grad_bout = _lib.ptr(lay.output_.weight.grad), _lib.ptr(lay.output_.bias.grad)
        if rules is not None:
            _lib.check(_lib.lib.dcll_conv_step_bwd_update_opt(ctypes.byref(desc), ctypes.byref(args), rules,
                                                              _lib.current_stream()))
            _store_optim(states[0], args.adam_i2h, rules[0])
            if lay.output_layer:
                _store_optim(states[1], args.adam_out, rules[1])
        else:
            _lib.check(_lib.lib.dcll_conv_step_bwd_update(ctypes.byref(desc), ctypes.byref(args), _lib.current_stream()))
            if fused:
                _store_steps(states[0], args.adam_i2h.step)
                if lay.output_layer:
                    _store_steps(states[1], args.adam_out.step)
            elif do_train:
                self.optimizer.step()                                   # ref:712
                if lay.output_layer:
                    self.optimizer2.step()                              # ref:714
        del keep
        return loss_t

    def _bwd_update_dense(self, target, do_train):
        lay = self.dclllayer
        (d, _ts, _wo, _bo, _x), outs = lay._ctx
        i2h = lay.i2h
        targ = _as_cuda_f32(target)
        dev = targ.device
        args = _lib.TrainArgs()
        kind = _step_loss_kind(self.crit, targ, outs['pvoutput'])
        args.loss_kind = kind
        keep = [targ]
        if kind == _lib.LOSS_EXTERNAL:
            pvo = outs['pvoutput'].detach().clone().requires_grad_(True)
            loss = self.crit(pvo, targ)
            loss.backward()
            keep.append(pvo.grad)
            args.g_o_ext = _lib.ptr(pvo.grad.contiguous())
            loss_t = loss.detach().reshape(1)
        else:
            args.target = _lib.ptr(targ)
            loss_t = self.crit(outs['pvoutput'], targ).detach().reshape(1)
        for p in (i2h.weight, i2h.bias):
            if p.grad is None or p.grad.shape != p.shape or not p.grad.is_contiguous():
                p.grad = torch.zeros_like(p)
        g_o = torch.empty((d.B, d.K), device=dev)
        g_u = torch.empty((d.B, d.Out), device=dev)
        d.g_o, d.g_u = _lib.ptr(g_o), _lib.ptr(g_u)
        d.grad_w, d.grad_b = _lib.ptr(i2h.weight.grad), _lib.ptr(i2h.bias.grad)
        fused = do_train and _is_plain_adam(self.optimizer)
        rule = _lib.Optim() if do_train and not fused and _device_optim(self.optimizer) is not None else None
        states = None
        if rule is not None:
            args.apply_update = 1
            states = _fill_optim(args.adam_i2h, rule, self.optimizer, i2h.weight, i2h.bias)
            _lib.check(_lib.lib.dcll_dense_step_bwd_update_opt(ctypes.byref(d), ctypes.byref(args), ctypes.byref(rule),
                                                               _lib.current_stream()))
            _store_optim(states, args.adam_i2h, rule)
        else:
            if fused:
                args.apply_update = 1
                states = _fill_adam(args.adam_i2h, self.optimizer, i2h.weight, i2h.bias)
            _lib.check(_lib.lib.dcll_dense_step_bwd_update(ctypes.byref(d), ctypes.byref(args), _lib.current_stream()))
            if fused:
                _store_steps(states, args.adam_i2h.step)
            elif do_train:
                self.optimizer.step()
        lay._g_u = g_u
        del keep
        return loss_t

    def train_dcll(self, input, target, do_train=True, regularize=0.05):
        """ref:690-718.  ``ConvNetwork.learn`` passes regularize=False, which is the implemented path."""
        if regularize:
            raise NotImplementedError('the activity regularisers (ref:698-701) are not implemented; '
                                      'every entry point passes regularize=False (networks/__init__.py:179)')
        output, pvoutput, pv, pvmem = self.forward(input)
        if self.iter >= self.burnin:
            tgt_loss = self._bwd_update(target, do_train)
        else:
            tgt_loss = torch.Tensor([0])
        return output, pvoutput, pv, pvmem, tgt_loss.detach()


class DCLLClassification(DCLLBase):
    def forward(self, input, ignore_burnin=False):                      # ref:722-729
        row = None
        if ignore_burnin or self.iter + 1 >= self.burnin:
            batch = input.shape[0]
            row = self.clout.next_row(int(batch))
        return super(DCLLClassification, self).forward(input, row)

    def write_stats(self, writer, label, epoch):                        # ref:731-733
        super(DCLLClassification, self).write_stats(writer, label, epoch)
        writer.add_scalar(self.name + '/acc/' + label, self.acc, epoch)

    def accuracy(self, targets):                                        # ref:735-738
        begin = len(self.clout)
        self.acc = accuracy_by_vote(self.clout, targets[-begin:])
        return self.acc

    def confusion_matrix(self, targets):                                # ref:740-749
        begin = len(self.clout)
        predictions_by_vote, labels_by_vote = get_predictions_by_vote(self.clout, targets[-begin:])
        num_classes = self.dclllayer.target_size
        confusion_matrix = np.zeros((num_classes, num_classes), dtype=int)
        for prediction, label in zip(predictions_by_vote, labels_by_vote):
            confusion_matrix[int(prediction), int(label)] += 1
        return confusion_matrix


def save_dcllslices(directory, slices):                                 # ref:789-791
    for i, s in enumerate(slices):
        torch.save(s.state_dict(), directory + '/slice_state{0}.pkl'.format(i))


def load_dcllslices(directory, slices):                                 # ref:794-797
    for i, s in enumerate(slices):
        s.load_state_dict(torch.load(directory + '/slice_state{0}.pkl'.format(i)))
