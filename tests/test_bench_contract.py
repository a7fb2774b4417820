"""bench.py's output contract on a machine without a GPU: the reference arm (`--impl reference`: the reference's own code from
the checkout named by DBOA_REFERENCE_ROOT through oracle/ref_harness.py, else the CPU port of the path) prints ONE JSON line
with the keys its readers rely on, and our own arm fails loudly instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), *args], capture_output=True, text=True, timeout=600, cwd=REPO,
                          env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_the_contract_line():
    r = run('--impl', 'reference', '--steps', '1', '--warmup', '0')
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
                'data', 'config', 'e2e', 'cpu_baseline', 'impl'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['unit'] == 'frames/s' and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['value'] > 0 and d['steps'] == 1 and d['gpu_launches'] == 0
    assert d['cpu_baseline']['kind'] in ('reference', 'port') and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_reference_arm_falls_back_to_the_port_without_a_reference_tree():
    r = run('--impl', 'reference', '--steps', '1', '--warmup', '0', env={'DBOA_REFERENCE_ROOT': 'none'})
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][0])
    assert d['cpu_baseline']['kind'] == 'port' and d['value'] > 0


def test_own_arm_needs_a_gpu_and_says_so():
    import torch
    if torch.cuda.is_available():
        return
    r = run('--steps', '1', '--warmup', '3')
    assert r.returncode != 0                                   # no silent CPU fallback
    assert 'cuda' in (r.stderr + r.stdout).lower()


def test_bad_arguments_are_refused(tmp_path):
    for args in (('--steps', '0'), ('--impl', 'reference', '--dump-outputs', str(tmp_path))):
        r = run(*args)
        assert r.returncode == 2 and 'error' in r.stderr, args
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_frame(tmp_path, asset_dir):
    """The dump is the prediction of the LAST timed frame: the same stream adapted frame by frame in this process (7 untimed
    prelude frames + 3 warm-up + 2 timed steps of bench.py, c2) and predicted after its last frame."""
    import torch
    from bench import WORKLOADS, default_options
    from conftest import rel_err
    from dynaboa_b200 import config, synthetic
    from dynaboa_b200.adaptor import Adaptor
    r = run('--steps', '2', '--warmup', '3', '--no-cpu-baseline', '--dump-outputs', str(tmp_path / 'out'))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][0])
    assert d['steps'] == 2
    n = 7 + 3 + 2
    opts = default_options(expdir=str(tmp_path), expname='ref', model_file=config.BASE_MODEL, synthetic_frames=n, rank=0, **WORKLOADS['c2'])
    ad = Adaptor(opts)
    ad.fused_eval = 'none'
    stream = synthetic.SyntheticStream(length=n, batch_size=1, rank=0)
    for t in range(n):
        ad.global_step, ad.fit_losses = t, {}
        batch = {k: stream[t][k].cuda() for k in ('image', 'smpl_j2d')}
        ad.adapt(batch)
    pred = ad.predict(batch['image'])
    torch.cuda.synchronize()
    first_timed = ad.predict(stream[n - 2]['image'].cuda())
    shapes = {'rotmat': (1, 24, 3, 3), 'betas': (1, 10), 'cam': (1, 3), 'joints': (1, 49, 3), 'vertices': (1, 6890, 3)}
    assert sorted(os.listdir(tmp_path / 'out')) == sorted(f'{k}.npy' for k in shapes)
    for k, shape in shapes.items():
        a = np.load(tmp_path / 'out' / f'{k}.npy')
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), k
        assert rel_err(a, pred[k]) < 1e-5, k
    assert rel_err(pred['vertices'], first_timed['vertices']) > 1e-3        # the frames are far enough apart to tell them apart
