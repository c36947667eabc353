"""The reference's real caller against the drop-in: `python VBx/vbhmm.py ...` unchanged (run_example.sh:23-34,
VBx/vbhmm.py:45,154-158), started through the launcher that makes `from VBx import VBx` resolve to vbx_b200.

The original VBx is not part of this repository; the tests that execute it read a checkout named by $VBX_REF.  So:
  * the import mechanics are tested everywhere with a two-directory mock (no GPU, no reference needed);
  * the unchanged vbhmm.py is executed where the reference exists: with a GPU it must reproduce exp/ES2005a.rttm, without
    one it must get through the reference's own I/O + AHC stages and then fail LOUDLY inside the drop-in (no CPU fallback);
  * what the drop-in computes for that exact call is covered on the GPU by tests/test_parity_gpu.py / test_pipeline.py.
"""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('VBX_REF', '')
SHIMS = os.path.join(ROOT, 'tests', 'shims')
GOLD = os.path.join(ROOT, 'tests', 'golden')


def reference_script():
    """The unmodified vbhmm.py: a checkout of the original VBx named by $VBX_REF, or a copy installed with
    `pip install --target baseline/_ref` from one (see DESIGN.md)."""
    for d in ([os.path.join(REF, 'VBx')] if REF else []) + [os.path.join(ROOT, 'baseline', '_ref', 'VBx')]:
        if os.path.isfile(os.path.join(d, 'vbhmm.py')) and os.path.isfile(os.path.join(d, 'VBx.py')):
            return os.path.join(d, 'vbhmm.py')
    return None


def _mock_tree(tmp_path):
    """A 'reference' directory with its own VBx.py next to the caller script, like VBx/VBx.py next to VBx/vbhmm.py."""
    d = tmp_path / 'refdir'
    d.mkdir()
    (d / 'VBx.py').write_text("def VBx(*a, **k):\n    raise SystemExit('the reference VBx.py was imported')\n")
    (d / 'helper_next_to_script.py').write_text('VALUE = 41\n')
    (d / 'caller.py').write_text(textwrap.dedent('''
        import sys
        from helper_next_to_script import VALUE          # siblings of the script must stay importable
        from VBx import VBx
        import VBx as module
        print('VBX_FROM', VBx.__module__, VALUE, sys.argv[1:], __name__, hasattr(module, 'forward_backward'), hasattr(module, 'DER'))
    '''))
    return d


def test_launcher_makes_the_shadow_module_win(tmp_path):
    d = _mock_tree(tmp_path)
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, '-m', 'vbx_b200.dropin.run', str(d / 'caller.py'), '--flag', 'x'],
                         capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    assert "VBX_FROM vbx_b200.api 41 ['--flag', 'x'] __main__ True True" in out.stdout


def test_pythonpath_alone_does_not_shadow_a_sibling_module(tmp_path):
    """Why the launcher exists: the script's directory is sys.path[0], ahead of PYTHONPATH."""
    d = _mock_tree(tmp_path)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, 'vbx_b200', 'dropin'), ROOT]))
    out = subprocess.run([sys.executable, str(d / 'caller.py')], capture_output=True, text=True, env=env, timeout=300)
    assert 'VBX_FROM VBx' in out.stdout          # the sibling VBx.py won


def test_shadow_module_exports_the_reference_names():
    import importlib
    m = importlib.import_module('vbx_b200.dropin.VBx')
    assert callable(m.VBx) and callable(m.forward_backward) and callable(m.DER)


@pytest.mark.gpu
@pytest.mark.skipif(reference_script() is None, reason='no copy of the original VBx ($VBX_REF or baseline/_ref)')
def test_unchanged_vbhmm_py_on_the_gpu_from_fixture_inputs(tmp_path):
    """On the GPU box: the UNCHANGED vbhmm.py (pip-installed copy of the reference) through the launcher, with its input
    files rebuilt from the reference-generated fixtures (x-vector ark, segments, binary Kaldi PLDA, transform) - the
    reference's own I/O, x-vector transform, AHC, softmax init, label merging and RTTM writer around OUR VBx().  The RTTM
    must equal the reference's system output for ES2005a (tests/golden/es2005a.npz) up to speaker renaming."""
    import numpy as np
    from vbx_b200 import formats
    z = np.load(os.path.join(GOLD, 'es2005a.npz'))
    m = np.load(os.path.join(GOLD, 'es2005a_model.npz'))
    keys, seg_lines = [], []
    for i, (s, e) in enumerate(z['seg_times']):
        k = f'ES2005a_{i:04d}-{int(round(s * 100)):08d}-{int(round(e * 100)):08d}'
        keys.append(k)
        seg_lines.append(f'{k} ES2005a {float(s)!r} {float(e)!r}')
    formats.write_vec_flt_ark(str(tmp_path / 'x.ark'), keys, z['x_raw'])
    (tmp_path / 'x.seg').write_text('\n'.join(seg_lines) + '\n')
    formats.write_kaldi_plda_binary(str(tmp_path / 'plda'), m['plda_mu'], m['plda_tr'], m['plda_psi'])
    np.savez(str(tmp_path / 'transform.npz'), mean1=m['mean1'], mean2=m['mean2'], lda=m['lda'])
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, SHIMS]))
    cmd = [sys.executable, '-m', 'vbx_b200.dropin.run', reference_script(),
           '--init', 'AHC+VB', '--out-rttm-dir', str(tmp_path / 'out'), '--xvec-ark-file', str(tmp_path / 'x.ark'),
           '--segments-file', str(tmp_path / 'x.seg'), '--xvec-transform', str(tmp_path / 'transform.npz'),
           '--plda-file', str(tmp_path / 'plda'), '--threshold', '-0.015', '--lda-dim', '128', '--Fa', '0.3', '--Fb', '17',
           '--loopP', '0.99']
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    got = formats.read_rttm(str(tmp_path / 'out' / 'ES2005a.rttm'))
    assert len(got) == len(z['rttm_starts'])
    mapping = {}
    for (r, s, d, lab), s2, e2, l2 in zip(got, z['rttm_starts'], z['rttm_ends'], z['rttm_labels']):
        assert r == 'ES2005a' and abs(s - s2) < 1e-5 and abs(d - (e2 - s2)) < 1e-5
        assert mapping.setdefault(lab, int(l2)) == int(l2)
    assert len(set(mapping.values())) == len(mapping)


@pytest.mark.skipif(not REF or not os.path.isfile(os.path.join(REF, 'VBx', 'vbhmm.py')),
                    reason='set VBX_REF to a checkout of the original VBx (its exp/ inputs are needed)')
def test_unchanged_vbhmm_py_through_the_dropin(tmp_path):
    import torch
    from vbx_b200 import formats
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, SHIMS]))
    cmd = [sys.executable, '-m', 'vbx_b200.dropin.run', os.path.join(REF, 'VBx', 'vbhmm.py'),
           '--init', 'AHC+VB', '--out-rttm-dir', str(tmp_path),
           '--xvec-ark-file', os.path.join(REF, 'exp', 'ES2005a.ark'), '--segments-file', os.path.join(REF, 'exp', 'ES2005a.seg'),
           '--xvec-transform', os.path.join(REF, 'VBx', 'models', 'ResNet101_16kHz', 'transform.h5'),
           '--plda-file', os.path.join(REF, 'VBx', 'models', 'ResNet101_16kHz', 'plda'),
           '--threshold', '-0.015', '--lda-dim', '128', '--Fa', '0.3', '--Fb', '17', '--loopP', '0.99']   # run_example.sh:23-34
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=900)
    assert 'ES2005a' in out.stdout                     # vbhmm.py:120 printed the recording name: I/O shims worked
    if not torch.cuda.is_available():
        # the reference's own stages ran (ark, h5, PLDA, AHC); the VB-HMM call reached vbx_b200 and refused to fall back
        assert out.returncode != 0
        assert 'no CUDA device - vbx_b200 has no CPU fallback' in out.stderr, out.stderr[-1500:]
        assert 'vbx_b200/api.py' in out.stderr
        return
    assert out.returncode == 0, out.stderr[-1500:]
    got = formats.read_rttm(str(tmp_path / 'ES2005a.rttm'))
    want = formats.read_rttm(os.path.join(REF, 'exp', 'ES2005a.rttm'))
    assert len(got) == len(want)
    mapping = {}
    for (r1, s1, d1, l1), (r2, s2, d2, l2) in zip(got, want):
        assert r1 == r2 and abs(s1 - s2) < 1e-5 and abs(d1 - d2) < 1e-5
        assert mapping.setdefault(l1, l2) == l2
    assert len(set(mapping.values())) == len(mapping)
