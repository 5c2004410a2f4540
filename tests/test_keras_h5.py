"""SURVEY.md 8 f1: Keras HDF5 weight files (pure-Python reader/writer, deephar_b200/hdf5.py + keras_h5.py)."""
import os

import numpy as np
import pytest

from deephar_b200 import hdf5, keras_h5, reception, spnet
from deephar_b200.config import ModelConfig, pa16j2d

HERE = os.path.dirname(os.path.abspath(__file__))
KW = dict(num_joints=4, dim=2, num_context_per_joint=2, num_blocks=1, ksize=(3, 3), concat_pose_confidence=False)


def test_hdf5_roundtrip_types_and_big_groups(tmp_path):
    p = str(tmp_path / 't.h5')
    rng = np.random.default_rng(0)
    data = {'g%d/d%03d' % (i % 3, i): rng.standard_normal((i % 5 + 1, 3)).astype(np.float32) for i in range(300)}
    with hdf5.Writer(p) as w:
        for k, v in data.items():
            w.create_dataset(k, v)
        w.create_dataset('ints', np.arange(7, dtype=np.int64))
        w.create_dataset('f64', np.linspace(0, 1, 5))
        w.create_dataset('scalar', np.float32(3.5))
        w.set_attr('/', 'names', np.array([b'alpha', b'be', b'gamma_long_name']))
        w.set_attr('/', 'version', '2.1.4')
        w.set_attr('g0', 'n', np.int32(42))
    with hdf5.File(p) as f:
        assert sorted(f.keys()) == ['f64', 'g0', 'g1', 'g2', 'ints', 'scalar']
        assert [s.decode() for s in f.attrs['names']] == ['alpha', 'be', 'gamma_long_name']
        assert f.attrs['version'] == b'2.1.4'
        assert int(f['g0'].attrs['n']) == 42
        assert len(f['g0'].keys()) == 100        # > one symbol-table node and > one B-tree level-0 node
        for k, v in data.items():
            np.testing.assert_array_equal(f[k].read(), v)
        np.testing.assert_array_equal(f['ints'].read(), np.arange(7))
        assert f['f64'].dtype == np.float64 and f['scalar'].read() == np.float32(3.5)
        with pytest.raises(KeyError):
            f['g0/nope']


def test_reads_a_file_written_by_libhdf5():
    """A file libhdf5 wrote: MATLAB v7.3 output from SciPy's test data, stored as tests/golden/testhdf5_7.4_GLNX86.mat
    (source and licence: testhdf5_7.4_GLNX86.mat.LICENSE beside it) -- 512-byte user block, old-style groups, v1 object
    headers, attributes."""
    path = os.path.join(HERE, 'golden', 'testhdf5_7.4_GLNX86.mat')
    with hdf5.File(path) as f:
        assert f.keys() == ['testdouble']
        d = f['testdouble']
        assert d.shape == (9, 1) and d.dtype == np.float64
        np.testing.assert_allclose(d.read()[:, 0], np.arange(9) * np.pi / 4, rtol=1e-12)
        assert d.attrs['MATLAB_class'] == b'double'


def test_not_hdf5_raises(tmp_path):
    p = tmp_path / 'x.h5'
    p.write_bytes(b'not an hdf5 file at all' * 10)
    with pytest.raises(hdf5.Hdf5Error):
        hdf5.File(str(p))


def test_save_load_weights_h5_roundtrip_reception(tmp_path):
    m = reception.build((32, 32, 3), **KW).init_synthetic_weights(3)
    p = str(tmp_path / 'weights_PE_test.h5')
    m.save_weights(p)
    # the file has the keras layout: nested sub-model groups, trainable weights before moving statistics
    with hdf5.File(p) as f:
        layers = [s.decode() for s in f.attrs['layer_names']]
        assert layers[:4] == ['Stem', 'rBlock1', 'SepConv1', 'RegMap1']
        wn = [s.decode() for s in f['Stem'].attrs['weight_names']]
        assert wn[0] == 'conv2d_1/kernel:0' and wn[-1].endswith('moving_variance:0') and 'moving' not in wn[len(wn) // 2 - 1]
    m2 = reception.build((32, 32, 3), **KW)
    m2.load_weights(p)                          # topological (by_name=False): everything must be there
    a, b = m.get_weights(), m2.get_weights()
    assert a.keys() == b.keys()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    assert m2.unused_file_weights == []


def test_load_by_name_partial_checkpoint_fixture():
    """tests/golden/tiny_keras_weights.h5 (written by make_h5_fixture.py): four stem layers + the frozen
    soft-argmax layers a real checkpoint carries."""
    path = os.path.join(HERE, 'golden', 'tiny_keras_weights.h5')
    m = reception.build((32, 32, 3), **KW).init_synthetic_weights(99)
    before = m.get_weights()
    with pytest.raises(KeyError):
        reception.build((32, 32, 3), **KW).load_weights(path)             # strict load of a partial file
    m.load_weights(path, by_name=True)
    after = m.get_weights()
    ref = reception.build((32, 32, 3), **KW).init_synthetic_weights(7).get_weights()
    changed = [k for k in after if not np.array_equal(after[k], before[k])]
    assert sorted(changed) == sorted(k for k in after if k.split('/')[0] == 'Stem' and
                                     k.split('/')[1] in ['%s_%d' % (p, i) for p in ('conv2d', 'batch_normalization')
                                                         for i in (1, 2, 3, 4)])
    for k in changed:
        np.testing.assert_array_equal(after[k], ref[k].astype(np.float16).astype(np.float32))
    assert sorted(set(g for g, _ in m.unused_file_weights)) == ['cSAM', 'sSAM']


def test_flat_and_timedistributed_names(tmp_path):
    """SPNet checkpoints have no sub-models: group = layer, variable '<layer>/<leaf>:0'; the CVPR'18 merge
    model wraps sub-models in TimeDistributed layers named 'td_<name>' (action.py:117-153)."""
    cfg = ModelConfig((2, 64, 64, 3), pa16j2d, num_actions=[5], num_pyramids=1, action_pyramids=[1], num_levels=2,
                      num_pose_features=16, num_visual_features=16, growth=32, image_div=8)
    m = spnet.build(cfg).init_synthetic_weights(5)
    p = str(tmp_path / 'spnet.hdf5')
    m.save_weights(p)
    m2 = spnet.build(cfg)
    m2.load_weights(p, by_name=True)
    for k, v in m.get_weights().items():
        np.testing.assert_array_equal(v, m2.get_weights()[k])
    assert keras_h5.candidates('td_Stem', 'conv2d_1/kernel:0')[0] == 'Stem/conv2d_1/kernel'
    assert 'conv1/kernel' in keras_h5.candidates('conv1', 'conv1/kernel:0')
    assert 'time_distributed_3/kernel' in keras_h5.candidates('time_distributed_3', 'time_distributed_3/kernel:0')


def test_shape_mismatch_is_an_error(tmp_path):
    m = reception.build((32, 32, 3), **KW).init_synthetic_weights(3)
    p = str(tmp_path / 'w.h5')
    m.save_weights(p)
    other = reception.build((32, 32, 3), **dict(KW, num_joints=5))
    with pytest.raises(ValueError):
        other.load_weights(p, by_name=True)


def test_damaged_files_raise_hdf5error_not_parser_internals(tmp_path):
    """Truncated downloads and flipped bytes: the reader either still finds a consistent file or raises hdf5.Hdf5Error
    (an IOError) -- never IndexError / struct noise, never a hang."""
    import random
    src = open(os.path.join(HERE, 'golden', 'tiny_keras_weights.h5'), 'rb').read()
    rnd = random.Random(7)
    p = str(tmp_path / 'damaged.h5')
    outcomes = {'ok': 0, 'error': 0}
    for it in range(240):
        b = bytearray(src)
        if it % 3 == 0:
            b = b[:rnd.randrange(1, len(b))]
        elif it % 3 == 1:
            for _ in range(rnd.randint(1, 4)):
                b[rnd.randrange(len(b))] = rnd.randrange(256)
        else:
            i = rnd.randrange(len(b) - 8)
            b[i:i + 8] = bytes([rnd.choice([0, 255])] * 8)
        with open(p, 'wb') as f:
            f.write(bytes(b))
        try:
            keras_h5.read_entries(p)
            outcomes['ok'] += 1
        except hdf5.Hdf5Error:
            outcomes['error'] += 1
    assert outcomes['error'] >= 80 and outcomes['ok'] >= 40          # every truncation fails; most flips hit float data
    with open(p, 'wb') as f:
        f.write(b'')
    with pytest.raises(hdf5.Hdf5Error):
        keras_h5.read_entries(p)
