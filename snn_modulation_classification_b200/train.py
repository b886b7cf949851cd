"""Training entry point: the reference's ``train.py`` CLI (ref train.py:17-95) on the B200 hot path.

Differences from the reference, all outside the hot path: the conventional baseline CNN
(``ReferenceConvNetwork``, ref train.py:199-202,256-260) is out of scope and not trained; without the RadioML
HDF5 file a synthetic loader with the same batch layout can be selected EXPLICITLY with ``--synthetic`` (a missing
``--radio_ml_data_dir`` is otherwise an error, as in the reference); tensorboardX is optional.  The hot loop (ref :249-251, :279-280) is one ``learn_window`` / ``test_window`` call.
"""
import argparse
import datetime
import os
import pickle

import numpy as np
import torch

from .data.utils import iq2spiketrain, to_one_hot
from .dcll.pytorch_libdcll import device
from .networks import ConvNetwork, load_network_spec


class _NullWriter:
    def __getattr__(self, name):
        return lambda *a, **k: None


def _writer(log_dir, comment):
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(log_dir=log_dir, comment=comment)
    except Exception:
        return _NullWriter()


def parse_args(argv=None):
    p = argparse.ArgumentParser(description='DCLL')
    p.add_argument('--data', type=str, default='RadioML', choices=['RadioML'], help='which data to use')
    p.add_argument('--radio_ml_data_dir', type=str, default='2018.01')
    p.add_argument('--synthetic', action='store_true',
                   help='use the synthetic RadioML-shaped stand-in loader (no data set needed); without this flag a '
                        'missing --radio_ml_data_dir is an error, as in the reference')
    p.add_argument('--min_snr', type=int, default=6)
    p.add_argument('--max_snr', type=int, default=30)
    p.add_argument('--per_h5_frac', type=float, default=0.5)
    p.add_argument('--train_frac', type=float, default=0.9)
    p.add_argument('--network_spec', type=str, default='networks/radio_ml_conv.yaml')
    p.add_argument('--ref_network_spec', type=str, default='networks/radio_ml_conv_ref.yaml')
    p.add_argument('--just_ref', action='store_true')
    p.add_argument('--I_resolution', type=int, default=128)
    p.add_argument('--Q_resolution', type=int, default=128)
    p.add_argument('--I_bounds', type=float, default=(-1, 1), nargs=2)
    p.add_argument('--Q_bounds', type=float, default=(-1, 1), nargs=2)
    p.add_argument('--restore_path', type=str)
    p.add_argument('--burnin', type=int, default=50)
    p.add_argument('--batch_size', type=int, default=64)
    p.add_argument('--batch_size_test', type=int, default=64)
    p.add_argument('--n_steps', type=int, default=10000)
    p.add_argument('--no_save', type=bool, default=False)
    p.add_argument('--seed', type=int, default=1)
    p.add_argument('--n_test_interval', type=int, default=20)
    p.add_argument('--n_test_samples', type=int, default=128)
    p.add_argument('--n_iters', type=int, default=1024)
    p.add_argument('--n_iters_test', type=int, default=1024)
    p.add_argument('--optim_type', type=str, default='Adam')
    p.add_argument('--loss_type', type=str, default='SmoothL1Loss')
    p.add_argument('--learning_rates', type=float, default=[1e-6], nargs='+')
    p.add_argument('--ref_lr', type=float, default=1e-3)
    p.add_argument('--alpha', type=float, default=.92)
    p.add_argument('--alphas', type=float, default=.85)
    p.add_argument('--alpharp', type=float, default=.65)
    p.add_argument('--arp', type=float, default=0)
    p.add_argument('--random_tau', type=bool, default=True)
    p.add_argument('--beta', type=float, default=.95)
    p.add_argument('--lc_ampl', type=float, default=0.5)
    p.add_argument('--netscale', type=float, default=1.)
    p.add_argument('--comment', type=str, default='')
    p.add_argument('--output', type=str, default='results')
    p.add_argument('--precision', type=str, default='fp32', choices=['fp32', 'bf16x3', 'f16x2'],
                   help="convolution arithmetic (ConvNetwork.set_precision): 'fp32' is FP32-exact, 'bf16x3' and 'f16x2' run "
                        "the tcgen05 tensor-core kernels where the layer shape has them")
    return p.parse_args(argv)


def get_loader(batch_size, train, synthetic=False, **kw):
    """The RadioML HDF5 reader (data/load_radio_ml.py) on ``data_dir``; the synthetic stand-in ONLY when asked for with
    ``--synthetic``.  A wrong path fails loudly (the reference does, data/load_radio_ml.py:69-71) instead of silently
    training and writing checkpoints on synthetic data."""
    if synthetic:
        from .data.synthetic import get_radio_ml_loader
        return get_radio_ml_loader(batch_size, train, **kw)
    data_dir = kw.get('data_dir')
    if not (data_dir and os.path.isdir(data_dir)):
        raise FileNotFoundError('--radio_ml_data_dir %r is not a directory (pass --synthetic for the synthetic '
                                'RadioML-shaped loader)' % (data_dir,))
    from .data.load_radio_ml import get_radio_ml_loader
    return get_radio_ml_loader(batch_size, train, **kw)


def main(argv=None):
    args = parse_args(argv)
    if args.just_ref:
        raise NotImplementedError('--just_ref trains the conventional baseline CNN, which is out of scope')
    torch.manual_seed(args.seed)                                        # ref :100-101
    np.random.seed(args.seed)
    current_time = datetime.datetime.now().strftime('%b%d_%H-%M-%S')
    log_dir = os.path.join('runs', args.data, current_time)
    writer = _writer(log_dir, '%s Conv' % args.data)
    out_dir = os.path.join(args.output, args.data, current_time)
    os.makedirs(out_dir, exist_ok=True)
    print('out dir: {out_dir}'.format(out_dir=out_dir))

    n_iters, n_iters_test = args.n_iters, args.n_iters_test
    im_dims = (1, args.Q_resolution, args.I_resolution)                 # ref :133
    target_size = 24
    loader_kw = dict(data_dir=args.radio_ml_data_dir, min_snr=args.min_snr, max_snr=args.max_snr,
                     per_h5_frac=args.per_h5_frac, train_frac=args.train_frac, synthetic=args.synthetic)
    st_kw = dict(out_w=args.I_resolution, out_h=args.Q_resolution, min_I=args.I_bounds[0], max_I=args.I_bounds[1],
                 min_Q=args.Q_bounds[0], max_Q=args.Q_bounds[1], gs_stdev=0, as_cells=True)
    n_test = int(np.ceil(float(args.n_test_samples) / args.batch_size_test))
    n_tests_total = int(np.ceil(float(args.n_steps) / args.n_test_interval))

    opt = getattr(torch.optim, args.optim_type)                         # ref :164-173
    opt_param = {'betas': [0.0, args.beta], 'weight_decay': 10.0}
    loss = getattr(torch.nn, args.loss_type)
    convs = load_network_spec(args.network_spec)
    net = ConvNetwork(args, im_dims, args.batch_size, convs, target_size, act=torch.nn.Sigmoid(), loss=loss, opt=opt,
                      opt_param=opt_param, learning_rates=args.learning_rates, burnin=args.burnin)
    if args.restore_path:                                               # ref :182-191
        if not os.path.isfile(args.restore_path):
            print('ERROR: Cannot load `%s`. File does not exist! Aborting load...' % args.restore_path)
        else:
            net.load_state_dict(torch.load(args.restore_path))
            print('Loaded the SNN model from `%s`.' % args.restore_path)
    net = net.to(device)
    net.reset(True)                                                     # ref :194 (only state zeroing)
    acc_test = np.empty([n_tests_total, n_test, len(net.dcll_slices)])

    if not args.no_save:
        with open(os.path.join(out_dir, 'args.txt'), 'w') as fp:
            fp.write(str(args))
        with open(os.path.join(out_dir, 'args.pkl'), 'wb') as fp:
            pickle.dump(vars(args), fp)

    train_data = get_loader(args.batch_size, train=True, **loader_kw)
    gen_train = iter(train_data)
    gen_test = iter(get_loader(args.batch_size_test, train=False, **loader_kw))
    all_test_data = [next(gen_test) for _ in range(n_test)]
    all_test_data = [(samples, to_one_hot(labels, target_size)) for (samples, labels) in all_test_data]

    label_train_counts = np.zeros(target_size, dtype=int)
    acc_train = None
    for step in range(args.n_steps):
        if ((step + 1) % 1000) == 0:                                    # ref :221-227
            for s in net.dcll_slices:
                s.optimizer.param_groups[-1]['lr'] /= 2
            net.dcll_slices[-1].optimizer2.param_groups[-1]['lr'] /= 2
            print('Adjusting learning rates')
        try:
            input, labels = next(gen_train)
        except StopIteration:
            gen_train = iter(train_data)
            input, labels = next(gen_train)
        for label in labels:
            label_train_counts[label] += 1
        labels = to_one_hot(labels, target_size)

        input_spikes, labels_spikes = iq2spiketrain(input, labels.to(device), max_duration=n_iters, **st_kw)
        net.reset()                                                     # ref :247-251
        net.train()
        net.learn_window(input_spikes, labels_spikes[0])
        acc_train = net.accuracy(labels_spikes)
        print('[TRAIN] Step {} \t Accuracy {}'.format(str(step).zfill(5), acc_train))

        if (step % args.n_test_interval) == 0:                          # ref :263-317
            test_idx = step // args.n_test_interval
            for i, test_data in enumerate(all_test_data):
                test_input, test_labels = iq2spiketrain(test_data[0], test_data[1].to(device),
                                                        max_duration=n_iters_test, **st_kw)
                net.reset()
                net.eval()
                net.test_window(test_input)
                acc_test[test_idx, i, :] = net.accuracy(test_labels)
                if i == 0:
                    net.write_stats(writer, step, comment='_batch_' + str(i))
            if not args.no_save:
                np.save(os.path.join(out_dir, 'acc_test.npy'), acc_test)
                save_path = os.path.join(out_dir, 'parameters_{}.pth'.format(step))
                torch.save({k: v.cpu() for k, v in net.state_dict().items()}, save_path)   # ref :300-303
                print('Saved network parameters to `%s`.' % save_path)
            acc = np.mean(acc_test[test_idx], axis=0)
            print('[TEST]  Step {} \t Accuracy {}'.format(str(step).zfill(5), acc))
    writer.close()
    return dict(out_dir=out_dir, acc_train=acc_train, acc_test=acc_test, net=net)


if __name__ == '__main__':
    main()
