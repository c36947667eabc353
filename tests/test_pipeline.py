"""The 'next' rows either side of the hot path (SURVEY.md 8f) against the ES2005a golden produced by the reference."""
import os

import numpy as np
import pytest
import torch

from vbx_b200 import pipeline

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(scope='module')
def es():
    return np.load(os.path.join(GOLD, 'es2005a.npz'))


def test_merge_adjacent_labels_matches_reference_output(es):
    s, e, l = pipeline.merge_adjacent_labels(es['seg_times'][:, 0], es['seg_times'][:, 1], es['labels'])
    np.testing.assert_allclose(s, es['rttm_starts'])
    np.testing.assert_allclose(e, es['rttm_ends'])
    assert np.array_equal(l, es['rttm_labels'])
    lines = pipeline.rttm_lines('ES2005a', s, e, l)
    assert lines[0] == 'SPEAKER ES2005a 1 0.000000 7.560000 <NA> <NA> %d <NA> <NA>' % (int(l[0]) + 1)
    assert len(lines) == 50


def test_merge_edge_cases():
    s, e, l = pipeline.merge_adjacent_labels([0.0, 1.0, 2.5, 2.6], [1.2, 2.0, 3.0, 4.0], np.array([0, 1, 1, 1]))
    np.testing.assert_allclose(s, [0.0, 1.1, 2.5])
    np.testing.assert_allclose(e, [1.1, 2.0, 4.0])
    assert l.tolist() == [0, 1, 1]
    s, e, l = pipeline.merge_adjacent_labels([], [], np.array([], dtype=int))
    assert len(s) == 0 and len(l) == 0


def test_soft_init_and_hard_labels_cpu(es):
    lab = torch.from_numpy(es['labels_ahc'].astype(np.int64))
    q = pipeline.soft_init(lab, int(lab.max()) + 1, float(es['smoothing']))
    assert torch.allclose(q.sum(1), torch.ones(len(lab)))
    assert torch.equal(q.argmax(1), lab)
    g = torch.from_numpy(es['gamma'])
    assert np.array_equal(pipeline.hard_labels(g).numpy(), es['labels'])
    a, b = pipeline.hard_labels(g, second=True)
    assert np.array_equal(b.numpy(), np.argsort(-es['gamma'], axis=1, kind='stable')[:, 1])


def test_xvector_transform_matches_reference_cpu(es):
    """VBx/vbhmm.py:129 (float64, CPU tensors here; the same code runs on the device), on the shipped ResNet101_16kHz
    model as stored in es2005a_model.npz.  Its PLDA is stored diagonalised (VBx/vbhmm.py:107-113: psi descending).
    The diagonalisation sees the model only through W = (tr' tr)^-1 and B = (tr' psi^-1 tr)^-1, which a permutation
    and sign flips of the rows of tr (with psi permuted alike) leave unchanged: from such a model it must recover the
    reference's order, signs and features."""
    m = np.load(os.path.join(GOLD, 'es2005a_model.npz'))
    assert str(m['sha_plda']) == str(es['sha_plda']) and str(m['sha_transform']) == str(es['sha_transform'])
    x = pipeline.xvector_transform(torch.from_numpy(es['x_raw'].astype(np.float64)), torch.from_numpy(m['mean1']),
                                   torch.from_numpy(m['mean2']), torch.from_numpy(m['lda']))
    np.testing.assert_allclose(x.numpy(), es['x_lda'], atol=1e-12)
    rng = np.random.default_rng(0)
    perm, sign = rng.permutation(len(m['plda_psi'])), rng.choice([-1.0, 1.0], size=len(m['plda_psi']))
    mu, tr, psi = pipeline.diagonalise_plda(m['plda_mu'], sign[:, None] * m['plda_tr'][perm], m['plda_psi'][perm])
    fea = pipeline.plda_project(x, torch.from_numpy(mu), torch.from_numpy(tr), 128)
    np.testing.assert_allclose(fea.numpy(), es['fea'], atol=1e-9)
    np.testing.assert_allclose(psi[:128], es['Phi'], rtol=1e-12)


@pytest.mark.gpu
def test_es2005a_rttm_end_to_end_on_gpu(es):
    """fea -> VB-HMM on the B200 -> labels -> merged segments == the reference's committed system output
    exp/ES2005a.rttm (50 segments, speaker ids up to renaming)."""
    from vbx_b200.batch import VbxBatch
    dev = torch.device('cuda:0')
    lab = torch.from_numpy(es['labels_ahc'].astype(np.int64)).to(dev)
    S = int(lab.max()) + 1
    T = len(lab)
    vb = VbxBatch([T], 128, S, device=dev)
    g = torch.zeros((T, vb.S), device=dev)
    g[:, :S] = pipeline.soft_init(lab, S, float(es['smoothing']))
    p = torch.zeros((1, vb.S), device=dev)
    p[0, :S] = 1.0 / S
    vb.prepare_scale(torch.from_numpy(es['fea'].astype(np.float32)).to(dev), torch.from_numpy(es['Phi'].astype(np.float32)).to(dev))
    vb.run(g, p, Fa=float(es['Fa']), Fb=float(es['Fb']), loopProb=float(es['loopProb']), maxIters=40, epsilon=1e-6)
    labels = pipeline.hard_labels(g[:, :S]).cpu().numpy()
    s, e, l = pipeline.merge_adjacent_labels(es['seg_times'][:, 0], es['seg_times'][:, 1], labels)
    np.testing.assert_allclose(s, es['rttm_starts'])
    np.testing.assert_allclose(e, es['rttm_ends'])
    mapping = {}
    for mine, ref in zip(l, es['rttm_ref_labels']):
        assert mapping.setdefault(int(mine), int(ref)) == int(ref)
    assert len(set(mapping.values())) == len(mapping) == 5
    vb.close()


@pytest.mark.gpu
def test_es2005a_raw_xvectors_to_rttm_on_gpu(es):
    """The whole real-data path on the device: raw x-vectors of exp/ES2005a.ark -> fused tcgen05 x-vector transform +
    PLDA projection (vbx_prepare_xvectors, VBx/vbhmm.py:125-129,153) -> VB-HMM -> RTTM, against the features and
    the system output the reference produces (tests/golden/make_golden.py)."""
    from vbx_b200.batch import VbxBatch
    m = np.load(os.path.join(GOLD, 'es2005a_model.npz'))
    assert str(m['sha_plda']) == str(es['sha_plda']) and str(m['sha_transform']) == str(es['sha_transform'])
    dev = torch.device('cuda:0')
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    T = es['x_raw'].shape[0]
    vb = VbxBatch([T], 128, 4, device=dev)
    rho, x_norm = vb.prepare_xvectors(f32(es['x_raw']), f32(m['mean1']), f32(m['lda']), f32(m['mean2']),
                                      f32(m['plda_mu']), f32(m['plda_tr']), f32(m['plda_psi']))
    torch.cuda.synchronize()
    # The shipped LDA matrix is badly conditioned (sum |a_k lda_kn| ~ 1000 x |sum|), so float32-level arithmetic shows:
    # numpy float32 reaches 3.9e-6 / 3.6e-5 on these two checks.  The operands are split three ways (exact, 6 MMAs), so what
    # is left is the float32 rounding of the model / inputs and the accumulation inside the tensor core (4x numpy's).
    e_x = np.abs(x_norm.double().cpu().numpy() - es['x_lda']).max()
    fea = rho.double().cpu().numpy() / np.sqrt(es['Phi'])[None, :]
    e_f = np.abs(fea - es['fea']).max()
    print('ES2005a chain: max |x_norm - ref| = %.2e, max |fea - ref| = %.2e (max |fea| = %.2f)' % (e_x, e_f, np.abs(es['fea']).max()))
    assert e_x <= 1.5e-5
    assert e_f <= 3e-4
    vb.close()
    lines, labels, g = pipeline.diarize_recording(
        es['x_raw'], es['seg_times'], es['labels_ahc'], (m['mean1'], m['mean2'], m['lda']),
        (m['plda_mu'], m['plda_tr'], m['plda_psi']), float(es['Fa']), float(es['Fb']), float(es['loopProb']),
        smoothing=float(es['smoothing']), max_iters=40, epsilon=1e-6, device=dev, recording='ES2005a',
        chain='tcgen05', plda_is_diagonal=True)
    assert np.array_equal(labels, es['labels'])
    e_g = np.abs(g.double().cpu().numpy() - es['gamma']).max()
    print('ES2005a chain: max |gamma - ref| = %.2e' % e_g)
    assert e_g <= 1e-4                       # the north-star bar, from raw x-vectors through both tensor-core passes
    assert len(lines) == 50 and all(l.startswith('SPEAKER ES2005a 1 ') for l in lines)
    starts = np.array([float(l.split()[3]) for l in lines])
    np.testing.assert_allclose(starts, es['rttm_starts'], atol=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize('chain', ['tcgen05', 'float64'])
def test_es2005a_everything_on_the_device(es, chain):
    """Raw x-vectors -> x-vector transform / PLDA projection -> AHC initialisation (vbx_ahc) -> VB-HMM -> labels, all
    on the B200; only the linkage matrix and the labels come back.  Equals the reference's AHC labels, final labels
    and RTTM segmentation."""
    m = np.load(os.path.join(GOLD, 'es2005a_model.npz'))
    dev = torch.device('cuda:0')
    lines, labels, g = pipeline.diarize_recording(
        es['x_raw'], es['seg_times'], None, (m['mean1'], m['mean2'], m['lda']),
        (m['plda_mu'], m['plda_tr'], m['plda_psi']), float(es['Fa']), float(es['Fb']), float(es['loopProb']),
        smoothing=float(es['smoothing']), max_iters=40, epsilon=1e-6, device=dev, recording='ES2005a',
        chain=chain, plda_is_diagonal=True, threshold=-0.015)
    assert g.shape[1] == es['gamma'].shape[1] == 31          # same AHC speaker count and numbering
    assert np.array_equal(labels, es['labels'])
    assert np.abs(g.double().cpu().numpy() - es['gamma']).max() <= 1e-4
    assert len(lines) == 50


@pytest.mark.gpu
def test_command_line_batch_of_recordings_to_rttm(tmp_path):
    """`python -m vbx_b200.cli` with the options of VBx/vbhmm.py on an archive holding TWO recordings (ES2005a twice under
    different names): Kaldi ark + segments + text PLDA + transform in, one RTTM per recording out, equal to the reference's
    exp/ES2005a.rttm up to speaker renaming."""
    from vbx_b200 import cli, formats
    z = np.load(os.path.join(GOLD, 'es2005a.npz'))
    m = np.load(os.path.join(GOLD, 'es2005a_model.npz'))
    T = z['x_raw'].shape[0]
    keys, seg_lines = [], []
    for rec in ('ES2005a', 'COPY0001'):
        for i, (s, e) in enumerate(z['seg_times']):
            k = f'{rec}_{i:04d}-{int(round(s * 100)):08d}-{int(round(e * 100)):08d}'
            keys.append(k)
            seg_lines.append(f'{k} {rec} {float(s)!r} {float(e)!r}')
    formats.write_vec_flt_ark(str(tmp_path / 'x.ark'), keys, np.concatenate([z['x_raw'], z['x_raw']]))
    (tmp_path / 'x.seg').write_text('\n'.join(seg_lines) + '\n')
    formats.write_kaldi_plda_text(str(tmp_path / 'plda.txt'), m['plda_mu'], m['plda_tr'], m['plda_psi'])
    np.savez(str(tmp_path / 'transform.npz'), mean1=m['mean1'], mean2=m['mean2'], lda=m['lda'])
    rc = cli.main(['--init', 'AHC+VB', '--out-rttm-dir', str(tmp_path / 'out'), '--xvec-ark-file', str(tmp_path / 'x.ark'),
                   '--segments-file', str(tmp_path / 'x.seg'), '--xvec-transform', str(tmp_path / 'transform.npz'),
                   '--plda-file', str(tmp_path / 'plda.txt'), '--threshold', '-0.015', '--lda-dim', '128', '--Fa', '0.3',
                   '--Fb', '17', '--loopP', '0.99', '--output-2nd', 'True'])
    assert rc == 0
    for rec in ('ES2005a', 'COPY0001'):
        got = formats.read_rttm(str(tmp_path / 'out' / f'{rec}.rttm'))
        assert len(got) == len(z['rttm_starts'])
        mapping = {}
        for (r, s, d, lab), s2, e2, l2 in zip(got, z['rttm_starts'], z['rttm_ends'], z['rttm_labels']):
            assert r == rec and abs(s - s2) < 1e-5 and abs(d - (e2 - s2)) < 1e-5
            assert mapping.setdefault(lab, int(l2)) == int(l2)
        assert len(set(mapping.values())) == len(mapping)
        assert os.path.exists(str(tmp_path / 'out2nd' / f'{rec}.rttm'))
