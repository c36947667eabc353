"""On-disk formats either side of the path (SURVEY.md 8f.4, App. B): the readers of vbx_b200/formats.py against byte
streams written here in the Kaldi layouts (kaldi_io.write_vec_flt at VBx/predict.py:193, Kaldi's Plda::Write)."""
import io
import os
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vbx_b200 import formats            # noqa: E402


def kaldi_vec(v, double=False):
    v = np.asarray(v, dtype='<f8' if double else '<f4')
    return (b'DV ' if double else b'FV ') + b'\x04' + struct.pack('<i', v.size) + v.tobytes()


def kaldi_mat(m, double=False):
    m = np.asarray(m, dtype='<f8' if double else '<f4')
    return (b'DM ' if double else b'FM ') + b'\x04' + struct.pack('<i', m.shape[0]) + b'\x04' + struct.pack('<i', m.shape[1]) + m.tobytes()


def test_ark_roundtrip_and_grouping(tmp_path):
    rng = np.random.default_rng(0)
    recs = {'ES2005a': 7, 'IS1009b_x': 3}
    path = tmp_path / 'x.ark'
    want = {}
    with open(path, 'wb') as f:
        for rec, n in recs.items():
            for i in range(n):
                key = f'{rec}_{i:04d}'
                v = rng.standard_normal(256).astype(np.float32)
                want.setdefault(rec, []).append(v)
                f.write(key.encode() + b' \0B' + kaldi_vec(v))
    got = formats.read_xvectors_by_recording(str(path))
    assert list(got) == list(recs)                      # archive order, recording id = key up to the last '_'
    for rec in recs:
        keys, x = got[rec]
        assert len(keys) == recs[rec] and x.shape == (recs[rec], 256)
        np.testing.assert_array_equal(x, np.array(want[rec]))


def test_ark_double_vectors_and_errors(tmp_path):
    path = tmp_path / 'd.ark'
    v = np.arange(5, dtype=np.float64) / 3
    with open(path, 'wb') as f:
        f.write(b'a_0 \0B' + kaldi_vec(v, double=True))
    (key, got), = list(formats.read_vec_flt_ark(str(path)))
    assert key == 'a_0'
    np.testing.assert_array_equal(got, v)
    bad = tmp_path / 'bad.ark'
    with open(bad, 'wb') as f:
        f.write(b'a_0 [ 1 2 3 ]\n')                     # text archives are not supported: loud error, no guess
    with pytest.raises(ValueError):
        list(formats.read_vec_flt_ark(str(bad)))


def test_segments(tmp_path):
    path = tmp_path / 'segments'
    path.write_text('ES2005a_0000 ES2005a 0.000 1.440\nES2005a_0001 ES2005a 0.240 1.680\n\nB_0 B 3.5 4.25\n')
    got = formats.read_segments(str(path))
    assert list(got) == ['ES2005a', 'B']
    names, times = got['ES2005a']
    assert names.tolist() == ['ES2005a_0000', 'ES2005a_0001']
    np.testing.assert_allclose(times, [[0.0, 1.44], [0.24, 1.68]])
    np.testing.assert_allclose(got['B'][1], [[3.5, 4.25]])


@pytest.mark.parametrize('double', [False, True])
def test_kaldi_plda(tmp_path, double):
    rng = np.random.default_rng(1)
    mean, tr, psi = rng.standard_normal(128), rng.standard_normal((128, 128)), rng.random(128) + 0.1
    path = tmp_path / 'plda'
    with open(path, 'wb') as f:
        f.write(b'\0B<Plda> ' + kaldi_vec(mean, double) + kaldi_mat(tr, double) + kaldi_vec(psi, double) + b'</Plda> ')
    m, t, p = formats.read_kaldi_plda(str(path))
    tol = 0 if double else 1e-6
    np.testing.assert_allclose(m, mean, rtol=tol, atol=tol)
    np.testing.assert_allclose(t, tr, rtol=tol, atol=tol)
    np.testing.assert_allclose(p, psi, rtol=tol, atol=tol)
    assert m.dtype == t.dtype == p.dtype == np.float64
    with open(path, 'wb') as f:
        f.write(b'\0B<Nnet> ')
    with pytest.raises(ValueError):
        formats.read_kaldi_plda(str(path))


def test_rttm_roundtrip(tmp_path):
    buf = io.StringIO()
    formats.write_rttm(buf, 'ES2005a', [0, 2, 0], [0.0, 1.5, 4.25], [1.5, 4.25, 6.0])
    lines = buf.getvalue().splitlines()
    assert lines[0] == 'SPEAKER ES2005a 1 0.000000 1.500000 <NA> <NA> 1 <NA> <NA>'       # VBx/vbhmm.py:48-51
    path = tmp_path / 'out.rttm'
    path.write_text(buf.getvalue())
    got = formats.read_rttm(str(path))
    assert [g[0] for g in got] == ['ES2005a'] * 3
    np.testing.assert_allclose([g[1] for g in got], [0.0, 1.5, 4.25])
    np.testing.assert_allclose([g[2] for g in got], [1.5, 2.75, 1.75])
    assert [g[3] for g in got] == ['1', '3', '1']


def test_transform_h5_rejects_other_files(tmp_path):
    path = tmp_path / 'transform.h5'
    path.write_bytes(b'\x89HDF\r\n\x1a\n' + b'\0' * 100)
    with pytest.raises(ValueError):
        formats.read_xvec_transform(str(path))


def test_shipped_model_files_when_present():
    """The readers on the model files shipped with the original VBx (a checkout named by $VBX_REF)."""
    ref_dir = os.path.join(os.environ.get('VBX_REF', ''), 'VBx', 'models', 'ResNet101_16kHz')
    if not os.environ.get('VBX_REF') or not os.path.exists(ref_dir):
        pytest.skip('set VBX_REF to a checkout of the original VBx to read its model files')
    m = np.load(os.path.join(ROOT, 'tests', 'golden', 'es2005a_model.npz'))
    mean1, mean2, lda = formats.read_xvec_transform(os.path.join(ref_dir, 'transform.h5'))
    np.testing.assert_array_equal(mean1, m['mean1'])
    np.testing.assert_array_equal(lda, m['lda'])
    mu, tr, psi = formats.read_kaldi_plda(os.path.join(ref_dir, 'plda'))
    np.testing.assert_array_equal(mu, m['plda_mu'])


def test_text_plda_round_trip_and_ark_writer(tmp_path):
    """Text-format Kaldi PLDA (VBx/kaldi_utils.py:41-48) and the ark writer used to build CLI fixtures."""
    from vbx_b200 import formats
    rng = np.random.default_rng(3)
    mean, tr, psi = rng.standard_normal(6), rng.standard_normal((6, 6)), np.sort(rng.uniform(0.1, 5, 6))[::-1].copy()
    f = str(tmp_path / 'plda.txt')
    formats.write_kaldi_plda_text(f, mean, tr, psi)
    m2, t2, p2 = formats.read_kaldi_plda(f)
    assert np.array_equal(mean, m2) and np.array_equal(tr, t2) and np.array_equal(psi, p2)
    assert open(f).read().startswith('<Plda>  [ ')
    with pytest.raises(ValueError):
        (tmp_path / 'bad.txt').write_text('<Nnet> [ 1 2 ]')
        formats.read_kaldi_plda(str(tmp_path / 'bad.txt'))
    keys = ['recA_0000-00000000-00000144', 'recA_0001-00000024-00000168', 'recB_0000-00000000-00000144']
    X = rng.standard_normal((3, 8)).astype(np.float32)
    ark = str(tmp_path / 'x.ark')
    formats.write_vec_flt_ark(ark, keys, X)
    got = formats.read_xvectors_by_recording(ark)
    assert list(got) == ['recA', 'recB'] and got['recA'][0] == keys[:2] and np.array_equal(got['recA'][1], X[:2])
    np.savez(str(tmp_path / 't.npz'), mean1=np.arange(4.0), mean2=np.arange(2.0), lda=np.ones((4, 2)))
    m1, m2_, lda = formats.read_xvec_transform(str(tmp_path / 't.npz'))
    assert m1.shape == (4,) and m2_.shape == (2,) and lda.shape == (4, 2)
