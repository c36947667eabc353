"""bench.py --dump-outputs: what it writes for a result of the timed path (float32 / float64 files within 64 MB, a
seeded frame sample of gamma that is the same on every call), the --steps check, and on the GPU that the files hold
the outputs of the timed path itself (against the float64 C oracle and the reference's ES2005a output)."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ('gamma_sample', 'gamma_sample_rows', 'pi', 'Li', 'n_iters', 'flags')


def load_bench():
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def fake_result(B, T, S_pad, iters, seed=0):
    g = torch.Generator().manual_seed(seed)
    out = dict(Li=torch.randn((B, iters), dtype=torch.float64, generator=g), n_iters=torch.full((B,), iters, dtype=torch.int32),
               flags=torch.zeros(B, dtype=torch.int32))
    return torch.rand((B * T, S_pad), generator=g), torch.rand((B, S_pad), generator=g), out


def check_dir(d, names):
    total = 0
    assert sorted(os.listdir(d)) == sorted(n + '.npy' for n in names)
    for n in names:
        a = np.load(os.path.join(d, n + '.npy'))
        assert a.dtype in (np.float32, np.float64), (n, a.dtype)
        total += os.path.getsize(os.path.join(d, n + '.npy'))
    assert total <= 64e6, total
    return {n: np.load(os.path.join(d, n + '.npy')) for n in names}


def test_dump_outputs_sample_types_and_size(tmp_path):
    bench = load_bench()
    gamma, pi, out = fake_result(B=300, T=500, S_pad=64, iters=4)      # gamma is 36 MB: sampled down to 32 MB
    trace = np.arange(8, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / 'a'), gamma, pi, out, 60, trace=trace)
    bench.dump_outputs(str(tmp_path / 'b'), gamma, pi, out, 60, trace=trace)
    a = check_dir(tmp_path / 'a', NAMES + ('elbo_trace',))
    b = check_dir(tmp_path / 'b', NAMES + ('elbo_trace',))
    for n in a:
        assert np.array_equal(a[n], b[n]), n
    rows = a['gamma_sample_rows'].astype(np.int64)
    assert len(rows) == (32 << 20) // (4 * 60) and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(a['gamma_sample'], gamma[rows, :60].numpy())
    np.testing.assert_array_equal(a['pi'], pi[:, :60].numpy())
    np.testing.assert_array_equal(a['Li'], out['Li'].numpy())
    np.testing.assert_array_equal(a['elbo_trace'], trace)


def test_row_indices_count_against_the_total(tmp_path):
    """S = 1: 32 MB of gamma would be 8.4 M rows and 67 MB of row indices; the sample shrinks to keep 64 MB in all."""
    bench = load_bench()
    gamma, pi, out = fake_result(B=6000, T=1000, S_pad=1, iters=2)
    bench.dump_outputs(str(tmp_path), gamma, pi, out, 1)
    a = check_dir(tmp_path, NAMES)
    assert 5_000_000 < len(a['gamma_sample_rows']) < 6_000_000


def test_small_output_is_dumped_whole(tmp_path):
    bench = load_bench()
    gamma, pi, out = fake_result(B=3, T=10, S_pad=8, iters=2)
    bench.dump_outputs(str(tmp_path), gamma, pi, out, 4)
    a = check_dir(tmp_path, NAMES)
    np.testing.assert_array_equal(a['gamma_sample'], gamma[:, :4].numpy())
    np.testing.assert_array_equal(a['gamma_sample_rows'], np.arange(30.0))


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and '--steps must be at least 1' in out.stderr


def run_bench(tmp_path, *args):
    d = str(tmp_path / 'dump')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *args, '--no-cpu-baseline', '--dump-outputs', d],
                         capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    return d


@pytest.mark.gpu
def test_dump_holds_the_timed_batch_outputs(tmp_path):
    """The synthetic batch of `--workload tiny` (all of gamma fits the dump), regenerated here from the same seeds, through
    the float64 C oracle: the dumped gamma, pi, Li and n_iters are those of the workload's 10 EM iterations."""
    from oracle import c_oracle
    bench = load_bench()
    d = check_dir(run_bench(tmp_path, '--workload', 'tiny', '--steps', '2', '--no-e2e', '--no-parity'), NAMES + ('elbo_trace',))
    w = bench.WORKLOADS['tiny']
    lens = bench.workload_lengths(w, seed=1000)
    data = bench.make_device_batch(lens, w['S'], seed=17, device=torch.device('cuda:0'))
    offs = np.concatenate([[0], np.cumsum(lens)])
    assert np.array_equal(d['gamma_sample_rows'], np.arange(offs[-1], dtype=np.float64))
    assert np.all(d['n_iters'] == w['iters'])
    V0, Phi = data['V0'].double().cpu().numpy(), data['Phi'].double().cpu().numpy()
    for b in (0, len(lens) // 2, len(lens) - 1):
        lo, hi = int(offs[b]), int(offs[b + 1])
        ref = c_oracle.vbx_oracle_batch(data['X'][lo:hi].double().cpu().numpy() @ V0, Phi, np.array([0, hi - lo]),
                                        data['gamma0'][lo:hi].double().cpu().numpy(), np.full(w['S'], 1.0 / w['S']),
                                        w['Fa'], w['Fb'], w['loopP'], w['iters'], -np.inf)
        assert np.abs(d['gamma_sample'][lo:hi] - ref['gamma']).max() <= 1e-4
        assert np.abs(d['pi'][b] - ref['pi'][0]).max() <= 1e-4
        np.testing.assert_allclose(d['Li'][b], ref['Li'][0], rtol=1e-4)


@pytest.mark.gpu
def test_dump_of_the_es2005a_call(tmp_path):
    """`--workload c1`: the timed device-resident run on ES2005a equals the reference's output for that call."""
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'es2005a.npz'))
    d = check_dir(run_bench(tmp_path, '--workload', 'c1', '--steps', '1'), NAMES)
    n = len(z['Li'])
    assert d['n_iters'].tolist() == [n]
    assert np.abs(d['gamma_sample'] - z['gamma']).max() <= 1e-4
    assert np.abs(d['pi'][0] - z['pi']).max() <= 1e-4
    np.testing.assert_allclose(d['Li'][0, :n], z['Li'], rtol=1e-4)
    assert np.all(np.isnan(d['Li'][0, n:]))
