"""RadioML reader (SURVEY section 8f, row N4): host logic of data/load_radio_ml.py on an in-memory HDF5 stand-in.

h5py and the 20 GB data set are not available, so the HDF5 module is replaced by a dictionary-backed fake with the four
calls the reader makes (File, create_dataset, item access, close).  When the original project is present (oracle/refshim.py
finds it), the reference's own RadioMLDataset runs on the SAME fake files and the two are compared element for
element; everywhere the interleave / split / layout properties are checked directly.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import refshim

REF = os.path.join(refshim.REFERENCE_ROOT, "data", "load_radio_ml.py")


class FakeH5:
    """Dictionary-backed stand-in for the h5py module; 'w' also touches the path so os.path.exists() sees the file."""

    def __init__(self):
        self.store = {}
        outer = self

        class File:
            def __init__(self, path, mode='r'):
                self.path, self.mode = path, mode
                if mode == 'w':
                    outer.store[path] = {}
                    open(path, 'wb').close()
                elif path not in outer.store:
                    raise OSError('no such file: %s' % path)

            def create_dataset(self, name, data):
                outer.store[self.path][name] = np.array(data)

            def __getitem__(self, name):
                return outer.store[self.path][name]

            def close(self):
                pass

        self.File = File


def _write_pairs(h5, data_dir, snrs, n_rec, seed=0):
    rs = np.random.RandomState(seed)
    for c in range(24):
        for z in snrs:
            f = h5.File(os.path.join(data_dir, 'class%d_snr%d.hdf5' % (c, z)), 'w')
            # value encodes (class, snr, record) so that misplaced records are visible, plus noise for min/max
            x = rs.randn(n_rec, 1024, 2).astype(np.float32) * 0.1
            x[:, 0, 0] = c
            x[:, 0, 1] = z
            x[:, 1, 0] = np.arange(n_rec)
            f.create_dataset('X', data=x)
            f.close()


def _reference_dataset_class(h5):
    if not os.path.isfile(REF):
        return None
    mod = types.ModuleType('h5py')
    mod.File = h5.File
    saved = sys.modules.get('h5py')
    sys.modules['h5py'] = mod
    try:
        spec = importlib.util.spec_from_file_location('_ref_load_radio_ml', REF)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
    finally:
        if saved is None:
            sys.modules.pop('h5py', None)
        else:
            sys.modules['h5py'] = saved
    return m.RadioMLDataset


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("normalize", [False, True])
def test_dataset_layout_split_and_interleave(tmp_path, train, normalize):
    from snn_modulation_classification_b200.data.load_radio_ml import RadioMLDataset
    h5 = FakeH5()
    d = str(tmp_path)
    snrs = [26, 28, 30]
    frac = 20 / 4096.0                                            # 20 records per pair, 18 train + 2 test
    _write_pairs(h5, d, snrs, n_rec=24)
    ds = RadioMLDataset(d, train, normalize=normalize, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9, h5=h5)
    per_pair = 18 if train else 2
    assert len(ds) == 24 * 3 * per_pair
    assert ds.X.shape == (len(ds), 2, 1, 1024) and ds.X.dtype == np.float32 and ds.Y.dtype == np.int64
    if not normalize:
        # global index n * 72 + (class * 3 + snr_index) holds record n (train) / 18 + n (test) of that pair
        for idx in (0, 1, 2, 3, 71, 72, 100, len(ds) - 1):
            slot, n = idx % 72, idx // 72
            c, zi = slot // 3, slot % 3
            x, y = ds[idx]
            assert y == c and x[0, 0, 0] == c and x[1, 0, 0] == snrs[zi] and x[0, 0, 1] == (n if train else 18 + n)
    else:
        assert float(ds.X.min()) >= 0.0 and float(ds.X.max()) <= 1.0
    ref_cls = _reference_dataset_class(h5)
    if ref_cls is not None:
        ref = ref_cls(d, train, normalize=normalize, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9)
        assert np.array_equal(ref.X, ds.X) and np.array_equal(ref.Y, ds.Y) and ref.X.dtype == ds.X.dtype


def test_gold_file_split_and_loader(tmp_path, capsys):
    from snn_modulation_classification_b200.data import load_radio_ml as L
    h5 = FakeH5()
    d = str(tmp_path)
    rs = np.random.RandomState(1)
    snr_all = list(range(-26, 32, 2))
    n = 24 * len(snr_all) * 2
    cls = np.repeat(np.arange(24), len(snr_all) * 2)
    z = np.tile(np.repeat(snr_all, 2), 24)
    f = h5.File(os.path.join(d, L.GOLD_FILE), 'w')
    x = rs.randn(n, 1024, 2).astype(np.float32)
    f.create_dataset('X', data=x)
    f.create_dataset('Y', data=np.eye(24, dtype=np.int64)[cls])
    f.create_dataset('Z', data=z[:, None].astype(np.int64))
    f.close()
    loader = L.get_radio_ml_loader(5, train=False, data_dir=d, min_snr=28, max_snr=30, per_h5_frac=2 / 4096.0, train_frac=0.5,
                                   h5=h5)
    assert os.path.exists(L.pair_file(d, 23, 30)) and loader.name == 'RadioML_test'
    assert len(loader.dataset) == 24 * 2 * 1
    xb, yb = next(iter(loader))
    assert xb.shape == (5, 2, 1, 1024) and xb.dtype == torch.float32 and yb.dtype == torch.int64      # ref :98-101
    # test split = second record of each pair, in (class, snr) order
    first = x[(cls == 0) & (z == 28)][1]
    assert np.array_equal(xb[0, :, 0, :].numpy(), first.T) and yb.tolist() == [0, 0, 1, 1, 2]
    ref_cls = _reference_dataset_class(h5)
    if ref_cls is not None:
        ref = ref_cls(d, True, min_snr=28, max_snr=30, per_h5_frac=2 / 4096.0, train_frac=0.5)
        mine = L.RadioMLDataset(d, True, min_snr=28, max_snr=30, per_h5_frac=2 / 4096.0, train_frac=0.5, h5=h5)
        assert np.array_equal(ref.X, mine.X) and np.array_equal(ref.Y, mine.Y)


def test_missing_files_fail_loudly(tmp_path):
    """Without h5py the install-free reader is used -- and an absent data set is still an error, never synthetic data."""
    from snn_modulation_classification_b200.data.load_radio_ml import RadioMLDataset
    with pytest.raises((OSError, IOError)):
        RadioMLDataset(str(tmp_path), True)


# ---------------------------------------------------------------------------------------------------------------------
# real files on disk: written by the test, read back through the install-free HDF5 reader (data/minih5.py)
# ---------------------------------------------------------------------------------------------------------------------
def test_minih5_file_structure_and_round_trip(tmp_path):
    """Byte-level checks of what the writer emits (HDF5 file-format specification, earliest format) + dtype round trips."""
    import struct
    from snn_modulation_classification_b200.data import minih5
    p = str(tmp_path / 'a.hdf5')
    rs = np.random.RandomState(0)
    x = rs.randn(7, 1024, 2).astype(np.float32)
    y = np.arange(12, dtype=np.int64).reshape(3, 4)
    z = rs.randn(5).astype(np.float64)
    f = minih5.File(p, 'w')
    f.create_dataset('X', data=x)
    f.create_dataset('Y', data=y)
    f.create_dataset('Z', data=z)
    f.close()
    raw = open(p, 'rb').read()
    assert raw[:8] == b'\x89HDF\r\n\x1a\n' and raw[8] == 0 and raw[13] == 8 and raw[14] == 8      # signature, superblock v0, 8-byte offsets
    eof = struct.unpack_from('<Q', raw, 40)[0]
    assert eof == len(raw)                                                                      # end-of-file address
    root_ohdr, cache = struct.unpack_from('<Q', raw, 64)[0], struct.unpack_from('<I', raw, 72)[0]
    btree, heap = struct.unpack_from('<QQ', raw, 80)
    assert raw[root_ohdr] == 1 and cache == 1 and raw[btree:btree + 4] == b'TREE' and raw[heap:heap + 4] == b'HEAP'
    snod = struct.unpack_from('<Q', raw, btree + 32)[0]
    assert raw[snod:snod + 4] == b'SNOD' and struct.unpack_from('<H', raw, snod + 6)[0] == 3
    assert raw.count(x.tobytes()) == 1 and raw.index(x.tobytes()) % 8 == 0                      # contiguous raw data, aligned
    g = minih5.File(p, 'r')
    assert sorted(g.keys()) == ['X', 'Y', 'Z'] and 'X' in g and 'W' not in g
    assert g['X'].shape == (7, 1024, 2) and g['X'].dtype == np.float32 and len(g['X']) == 7
    assert np.array_equal(g['X'][:], x) and np.array_equal(g['X'][2:5], x[2:5]) and np.array_equal(g['X'][:, 3, 1], x[:, 3, 1])
    assert np.array_equal(g['Y'][:], y) and g['Y'].dtype == np.int64 and np.array_equal(np.argmax(g['Y'], axis=1), np.argmax(y, axis=1))
    assert np.array_equal(g['Z'][:], z) and g['Z'].dtype == np.float64
    with pytest.raises(KeyError):
        g['W']
    g.close()
    open(str(tmp_path / 'b.hdf5'), 'wb').write(b'not hdf5 at all' * 10)
    with pytest.raises(IOError):
        minih5.File(str(tmp_path / 'b.hdf5'), 'r')


@pytest.mark.parametrize("train", [True, False])
def test_loader_reads_real_files_on_disk(tmp_path, train):
    """RadioMLDataset over per-(class, SNR) HDF5 files that exist on disk (72 files written by the test), through whichever HDF5
    module the loader finds (h5py if installed, else data/minih5.py) -- same contents as over the in-memory stand-in, and as the
    reference class when it is present."""
    from snn_modulation_classification_b200.data import load_radio_ml as L
    from snn_modulation_classification_b200.data import minih5
    d = str(tmp_path)
    snrs = [26, 28, 30]
    frac = 20 / 4096.0
    _write_pairs(minih5, d, snrs, n_rec=24)
    assert os.path.getsize(L.pair_file(d, 5, 28)) > 24 * 1024 * 2 * 4
    ds = L.RadioMLDataset(d, train, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9)          # h5 = None: auto-select
    fake = FakeH5()
    os.makedirs(str(tmp_path / 'fake'))
    _write_pairs(fake, str(tmp_path / 'fake'), snrs, n_rec=24)
    want = L.RadioMLDataset(str(tmp_path / 'fake'), train, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9, h5=fake)
    assert np.array_equal(ds.X, want.X) and np.array_equal(ds.Y, want.Y) and ds.X.dtype == np.float32
    loader = L.get_radio_ml_loader(6, train=train, data_dir=d, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9)
    xb, yb = next(iter(loader))
    assert xb.shape == (6, 2, 1, 1024) and xb.dtype == torch.float32 and yb.dtype == torch.int64
    ref_cls = _reference_dataset_class(minih5)
    if ref_cls is not None:                               # the reference's own class reading the same on-disk files
        ref = ref_cls(d, train, min_snr=26, max_snr=30, per_h5_frac=frac, train_frac=0.9)
        assert np.array_equal(ref.X, ds.X) and np.array_equal(ref.Y, ds.Y)
