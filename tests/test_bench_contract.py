"""bench.py contract checks: the reference arm prints one JSON line with the agreed keys, `--precision auto` resolves per net, the f8
numerics model stays where the design says (3-4 % of the single-pass fp16 error), and `--dump-outputs` writes what the last timed step
returned (the native arm's check needs a GPU, the others do not)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def _run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--cpu_batch', '2',
                          '--num_steps', '3'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype', 'data',
              'config', 'impl', 'cpu_baseline', 'e2e'):
        assert k in line, k
    assert line['impl'] == 'reference' and line['value'] > 0 and line['higher_is_better'] is True and line['vs_baseline'] is None
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1 and line['cpu_baseline']['value'] == line['value']
    assert line['e2e'] == dict(value=line['value'], unit=line['unit'], h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert 'workload' in line['config'] and 'model' not in line['config']


def test_precision_auto_resolves_per_net(monkeypatch):
    bench = _bench_module()
    for net, want, fmin in (('cifar10', 'fp16f8', 0), ('imagenet64', 'fp16f8', 0), ('ffhq', 'fp16f8', 256), ('sd15', bench.PRECISION_FOR['sd15'], 0)):
        monkeypatch.setattr(sys, 'argv', ['bench.py', '--net', net])
        a = bench.parse()
        assert (a.precision, a.precision_requested, a.f8_min_channels) == (want, 'auto', fmin)
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--net', 'ffhq', '--precision', 'fp16f8'])
    a = bench.parse()
    assert a.precision == 'fp16f8' and a.f8_min_channels == 0          # an explicit precision keeps f8_min_channels as given


def test_f8_operand_model_error_budget():
    """CPU emulation of the operand formats of the f8 GEMM mode inside the oracle (tests/study_fp8_corrections.py): the denoiser error
    is a few percent of the single-pass fp16 error and well inside 1e-3 on the de-zeroed reduced-size nets."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import study_fp8_corrections as St
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    for name in ('tiny_song', 'tiny_adm'):
        r = {k: max(v) for k, v in St.run(name, batch=2, sigmas=(80.0, 0.5)).items()}
        assert r['fp16x3'] < 2e-5 and r['fp16+f8'] < 2e-4
        assert r['fp16+f8'] < 0.08 * r['fp16'], r


def test_steps_must_be_positive(monkeypatch):
    bench = _bench_module()
    for steps in ('0', '-1'):
        monkeypatch.setattr(sys, 'argv', ['bench.py', '--steps', steps])
        with pytest.raises(SystemExit):
            bench.parse()


def test_reference_arm_dumps_its_last_timed_step(tmp_path):
    """The reference arm's timed path is the oracle sampler: the dump is its output on the bench's fixed latents."""
    from oracle import edm_oracle as O
    from oracle import solvers_oracle as SO
    line = _run_bench('--impl', 'reference', '--steps', '2', '--warmup', '0', '--cpu_batch', '2', '--num_steps', '3', '--dump-outputs', str(tmp_path))
    assert line['steps'] == 2
    assert os.listdir(tmp_path) == ['samples.npy']
    got = np.load(tmp_path / 'samples.npy')
    P, S = O.make_net('cifar10', seed=0, dezero=True)
    want = SO.sample(O.OracleNet(P, S), O.stacked_randn(range(2), (3, 32, 32)), 'heun', num_steps=3).detach().numpy()
    assert got.dtype == np.float32 and got.shape == want.shape == (2, 3, 32, 32)
    assert np.allclose(got, want, rtol=0, atol=1e-5)


def test_dump_keeps_a_seeded_sample_within_the_limit(tmp_path, monkeypatch):
    bench = _bench_module()
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 4096)
    arrays = dict(a=torch.arange(80 * 16, dtype=torch.float64).reshape(80, 16), b=torch.randn(10, 3, 8))      # 5120 + 960 bytes as float32
    files = []
    for run in ('1', '2'):
        bench.write_outputs(str(tmp_path / run), arrays)
        files.append({k: np.load(tmp_path / run / f'{k}.npy') for k in arrays})
    a, b = files[0]['a'], files[0]['b']
    assert a.dtype == b.dtype == np.float32 and a.nbytes + b.nbytes <= 4096 and len(a) > 40 and len(b) > 4
    rows = a[:, 0].astype(int) // 16
    assert (np.diff(rows) > 0).all() and np.array_equal(a, arrays['a'].numpy()[rows])    # whole rows of the array, in order
    assert all(np.array_equal(files[0][k], files[1][k]) for k in arrays)                  # the same sample every run
    bench.write_outputs(str(tmp_path / 'small'), dict(b=arrays['b']))
    assert np.array_equal(np.load(tmp_path / 'small' / 'b.npy'), arrays['b'].numpy())     # under the limit: everything


@pytest.mark.gpu
def test_native_arm_dumps_its_last_timed_step(tmp_path, monkeypatch):
    """The native arm's dump is the final images of its last timed sampling pass: the same sampler on the bench's own seeded workload,
    run again in this process, gives the same images."""
    args = ['--steps', '2', '--warmup', '1', '--batch', '2', '--num_steps', '3', '--no_extras', '--no_cpu_baseline']
    line = _run_bench(*args, '--dump-outputs', str(tmp_path))
    assert line['steps'] == 2 and line['gpu_launches'] > 0
    assert os.listdir(tmp_path) == ['samples.npy']
    got = np.load(tmp_path / 'samples.npy')
    bench = _bench_module()
    monkeypatch.setattr(sys, 'argv', ['bench.py', *args])
    net, sampler, kw, latents, _ = bench.build_workload(bench.parse(), torch.device('cuda', 0), 0)
    want = sampler(net, latents, **kw).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == want.shape == (2, 3, 32, 32)
    assert np.abs(got - want).max() <= 1e-5 and np.abs(got - latents.cpu().numpy()).max() > 0.1
